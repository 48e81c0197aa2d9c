// nve.cu -- the repo's own velocity-Verlet harness around the cavity force (NOT HOOMD's integrator; HOOMD's
// TwoStepConstantVolume is upstream code that is not in the reference tree).  Everything here uses the arithmetic of
// oracle/cavity_oracle.c orc_nve_step / orc_nvt_step: hm = 0.5*dt/m; v = v + hm*f; r = r + dt*v, each product and sum
// rounded separately (no FMA) so that both arms integrate identically.  In order of increasing fusion:
//   k_nve<DRIFT>            cavb200_nve_kick_drift / _half_kick: plain NVE steps (energy-drift comparison)
//   k_nvt_one / k_nvt_two   SURVEY.md 8f.1: the Bussi rescale rides on the first half step, the kinetic energy for the
//                           NEXT step is summed while the second half step writes the velocities (no thermostat pass)
//   ... <RANK1>             SURVEY.md 8f.2: the cavity force is never stored, F_i = (-g c_i) Dq is formed in the kick
//   k_net_force_add_rank1   what a net-force sum does with that rank-1 contribution
//   k_md_one                step one with the NEXT force's dipole reduce inside (positions read once)
//   k_md_fused              step two of step t-1 + step one of step t in ONE persistent launch (148 B/particle)
//   ... <MASK>              the thermostatted group as the handle's bit mask instead of a window (cavb200_group_set)
//   k_group_mask / k_photon_reindex   cavb200_group_set / cavb200_rank1_reindex (once per particle sort)
#include "hotpath.cuh"

#include <type_traits>

#ifndef CAVB_NVT_CTAS_PER_SM
#define CAVB_NVT_CTAS_PER_SM 4 // grid cap of the element-wise harness kernels, in CTAs of 256 threads per SM: one wave (A/B at 1M: 8 -> 4: path C 55.7 -> 51.4 us, D 48.6 -> 44.7 us)
#endif

namespace cavb
    {
// step one: alpha from the KE left in Scalars by the previous step two (or by cavb200_bussi_ke);
// group: v <- alpha v;  all: v += dt/2 f/m;  r += dt v.  Purely element-wise: no hand-off.
// RANK1 (SURVEY.md 8f.2): the cavity force is never stored -- it is rank-1, F_i = (-g c_i) Dq
// (reference src/CavityForceCompute.cc:188-200), so the kick forms it from the charge and the Final
// record cavb200_force_rank1 left on the device and adds it to the other forces (force may be NULL).
struct Rank1In
    {
    const double* charge;
    const Final* fin;
    ForceIn f; // pos (type look-up, only when several 'L' particles exist), L_typeid, g
    };

// Box wrap of the drift (SURVEY.md 8a row a11: r <- r + v dt, wrap): HOOMD's BoxDim::wrap for an orthorhombic box that is
// periodic in all three directions, [-L/2, L/2) -- one shift per direction, the image flag follows
// [HOOMD-upstream, not in the reference tree: restated from its definition; oracle: orc_wrap].
__device__ __forceinline__ bool wrap_one(double& x, int& img, double L, double hi)
    {
    if (x >= hi)
        {
        x = __dadd_rn(x, -L);
        img++;
        return true;
        }
    if (x < -hi)
        {
        x = __dadd_rn(x, L);
        img--;
        return true;
        }
    return false;
    }
struct WrapIn
    {
    int* image; // int3 per particle, read and (when a particle crosses a face) written
    double Lx, Ly, Lz;
    };
// wrap p and keep the particle's image flags in step; returns the (new) flags
__device__ __forceinline__ void wrap_particle(double4& p, unsigned long long i, const WrapIn& w, int& ix, int& iy, int& iz)
    {
    bool ch = wrap_one(p.x, ix, w.Lx, __dmul_rn(0.5, w.Lx));
    ch = wrap_one(p.y, iy, w.Ly, __dmul_rn(0.5, w.Ly)) || ch;
    ch = wrap_one(p.z, iz, w.Lz, __dmul_rn(0.5, w.Lz)) || ch;
    if (ch)
        {
        w.image[3 * i + 0] = ix;
        w.image[3 * i + 1] = iy;
        w.image[3 * i + 2] = iz;
        }
    }

// Membership of the thermostatted group: the window [lo, hi), or (MASK) bit i of the handle's group mask
// (cavb200_group_set: ceil(N/32) words, bit i%32 of word i/32).  Every launch of these kernels has a block size and a
// grid stride that are multiples of 32, so the lanes of a warp hold 32 consecutive indices and read ONE mask word, a
// broadcast load: 4 B per 32 particles and pass.
// (Written out at each test as `MASK ? in_mask(mask, i) : i >= lo && i < hi`: behind a helper function returning bool
// the window test compiles to different, if equivalent, instructions.)
__device__ __forceinline__ bool in_mask(const uint32_t* mask, unsigned long long i)
    {
    return (__ldg(mask + (i >> 5)) >> (i & 31)) & 1u;
    }

// v += hm f and r += dt v, each product and sum rounded separately (hm = dt/2 / m)
__device__ __forceinline__ void half_kick(double4& v, double hm, const double4& f)
    {
    v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
    v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
    v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
    }
__device__ __forceinline__ void drift(double4& p, double dt, const double4& v)
    {
    p.x = __dadd_rn(p.x, __dmul_rn(dt, v.x));
    p.y = __dadd_rn(p.y, __dmul_rn(dt, v.y));
    p.z = __dadd_rn(p.z, __dmul_rn(dt, v.z));
    }

// fc += fo: the other forces added to the rank-1 cavity force fc; the potential-energy slot is theirs, the cavity term's
// is 0 (:145,180)
__device__ __forceinline__ void add_other(double4& fc, const double4& fo)
    {
    fc.x = __dadd_rn(fo.x, fc.x);
    fc.y = __dadd_rn(fo.y, fc.y);
    fc.z = __dadd_rn(fo.z, fc.z);
    fc.w = fo.w;
    }

// The kick force of particle i with charge c: the rank-1 cavity force, plus the other forces when force_other is given
__device__ __forceinline__ double4 rank1_force(const double4* force_other, unsigned long long i, double c, const Rank1In& r,
                                               const Final& fin)
    {
    double4 f = force_of(i, c, fin, r.f);
    if (force_other)
        add_other(f, ld256(force_other + i));
    return f;
    }

template<bool RANK1>
__device__ __forceinline__ double4 kick_force(const double4* force, unsigned long long i, const Rank1In& r, const Final& fin)
    {
    if (!RANK1)
        return ld256(force + i);
    return rank1_force(force, i, __ldg(r.charge + i), r, fin);
    }

// Image flags of particle i.  WRAP: the kernel rewrites them, so they are read coherently, not through the read-only path.
template<bool WRAP>
__device__ __forceinline__ int3 load_image(const WrapIn& w, const int* image, unsigned long long i)
    {
    if (WRAP)
        return make_int3(w.image[3 * i + 0], w.image[3 * i + 1], w.image[3 * i + 2]);
    return make_int3(__ldg(image + 3 * i + 0), __ldg(image + 3 * i + 1), __ldg(image + 3 * i + 2));
    }

// Step one's thermostat prologue, run by thread 0 of every CTA: alpha from the KE that the previous step two (or
// cavb200_bussi_ke) left in Scalars, 1 without a rescale; CTA 0 also keeps the reservoir books.
__device__ __forceinline__ double step_one_alpha(const BussiIn& b, Scalars* scalars)
    {
    double alpha = 1.0;
    if (b.rescale && b.n > 0)
        {
        int ok = 1;
        const double KE = scalars->ke;
        alpha = bussi_alpha(KE, b, ok);
        if (blockIdx.x == 0)
            {
            if (ok)
                {
                // BussiReservoirThermostat.h:86-95
                const double inst = __dmul_rn(KE, __dadd_rn(1.0, -__dmul_rn(alpha, alpha)));
                scalars->alpha = alpha;
                scalars->inst = inst;
                scalars->cumulative = __dadd_rn(scalars->cumulative, inst);
                }
            scalars->err = ok ? 0.0 : 1.0; // 1: zero kinetic energy with dof != 0 (:57-61), no rescale
            }
        }
    return alpha;
    }

// Thread 0 publishes the CTA's record and takes a ticket; true in every thread of the last CTA to take one, which then
// folds the records (fixed order) and resets the ticket.
__device__ __forceinline__ bool last_to_publish(Partial* recs, const BlockScratch& sc, unsigned long long* ticket, int& s_last)
    {
    if (threadIdx.x == 0)
        {
        publish_record(recs + blockIdx.x, sc.rec, 0ull);
        __threadfence();
        const unsigned long long t = atom_acq_rel_add_u64(ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
        }
    __syncthreads();
    return s_last;
    }

template<bool RANK1, bool WRAP, bool MASK>
__global__ void __launch_bounds__(256)
    k_nvt_one(double4* pos, double4* vel, const double4* force, uint32_t N, double dt, BussiIn b, Scalars* scalars,
              Rank1In r1, WrapIn w, const uint32_t* mask)
    {
    __shared__ double s_alpha;
    __shared__ Final s_fin;
    if (threadIdx.x == 0)
        {
        if (RANK1)
            s_fin = *r1.fin;
        s_alpha = step_one_alpha(b, scalars);
        }
    __syncthreads();
    const double alpha = s_alpha;
    const unsigned long long lo = b.first, hi = (unsigned long long)b.first + b.n;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        {
        double4 v = ld256(vel + i);
        const double4 f = kick_force<RANK1>(force, i, r1, s_fin);
        double4 p = ld256(pos + i);
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            {
            v.x = __dmul_rn(v.x, alpha);
            v.y = __dmul_rn(v.y, alpha);
            v.z = __dmul_rn(v.z, alpha);
            }
        half_kick(v, __ddiv_rn(__dmul_rn(0.5, dt), v.w), f);
        drift(p, dt, v);
        if (WRAP)
            {
            int ix = w.image[3 * i + 0], iy = w.image[3 * i + 1], iz = w.image[3 * i + 2];
            wrap_particle(p, i, w, ix, iy, iz);
            }
        st256(vel + i, v);
        st256(pos + i, p);
        }
    }

// step two: all: v += dt/2 f/m, and sum m|v|^2 of the group on the way out; the last CTA to take a
// ticket folds the CTA records (fixed order) and leaves KE in Scalars for the next step one.
template<bool RANK1, bool MASK>
__global__ void __launch_bounds__(256)
    k_nvt_two(double4* vel, const double4* force, uint32_t N, double dt, BussiIn b, Partial* recs, Scalars* scalars,
              unsigned long long* ticket, Rank1In r1, const uint32_t* mask)
    {
    __shared__ BlockScratch sc;
    __shared__ int s_last;
    __shared__ Final s_fin;
    if (threadIdx.x == 0)
        {
        sc.flags = 0u;
        if (RANK1)
            s_fin = *r1.fin;
        }
    if (RANK1)
        __syncthreads();
    Acc a;
    acc_zero(a);
    const unsigned long long lo = b.first, hi = (unsigned long long)b.first + b.n;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        {
        double4 v = ld256(vel + i);
        const double4 f = kick_force<RANK1>(force, i, r1, s_fin);
        half_kick(v, __ddiv_rn(__dmul_rn(0.5, dt), v.w), f);
        st256(vel + i, v);
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            a.ke += v.w * (v.x * v.x + v.y * v.y + v.z * v.z);
        }
    ForceIn f0 = {};
    block_merge<false, true>(a, f0, sc);
    if (!last_to_publish(recs, sc, ticket, s_last))
        return;
    BussiIn ke_only = b;
    ke_only.rescale = 0; // finalize: Scalars.ke = 1/2 sum, nothing else
    combine_phase<false, true, false, true>(recs, (int)gridDim.x, 0ull, f0, ke_only, sc, scalars, true);
    if (threadIdx.x == 0)
        *ticket = 0ull;
    }

// Step one of the thermostatted harness with the NEXT cavity force's reduce pass folded in (SURVEY.md 8f.1 + 8f.2):
// the kick uses the rank-1 force of the previous Final record, the drift produces the new position, and the
// dipole term charge * (r_new + image L) of that new position is accumulated on the spot
// (src/CavityForceCompute.cc:107-109,124) -- positions are never read a second time.  The last CTA to take a
// ticket folds the CTA records and leaves the new Scalars / Final for step two.  One launch replaces
// cavb200_nvt_step_one_rank1 + cavb200_force_rank1.
template<bool WRAP, bool MASK>
__global__ void __launch_bounds__(256, 3)
    k_md_one(double4* pos, double4* vel, const double4* force_other, uint32_t N, double dt, BussiIn b, Scalars* scalars,
             Rank1In r1, ForceIn fnew, Partial* recs, unsigned long long* ticket, Final* fin_out, WrapIn w,
             const uint32_t* mask)
    {
    __shared__ BlockScratch sc;
    __shared__ double s_alpha;
    __shared__ Final s_fin;
    __shared__ int s_last;
    if (threadIdx.x == 0)
        {
        sc.flags = 0u;
        s_fin = *r1.fin;
        s_alpha = step_one_alpha(b, scalars);
        }
    __syncthreads();
    const double alpha = s_alpha;
    const unsigned long long lo = b.first, hi = (unsigned long long)b.first + b.n;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    Acc a;
    acc_zero(a);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        {
        double4 v = ld256(vel + i);
        double4 p = ld256(pos + i);
        const double c = __ldg(fnew.charge + i);
        int3 im = load_image<WRAP>(w, fnew.image, i);
        const double4 f = rank1_force(force_other, i, c, r1, s_fin);
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            {
            v.x = __dmul_rn(v.x, alpha);
            v.y = __dmul_rn(v.y, alpha);
            v.z = __dmul_rn(v.z, alpha);
            }
        half_kick(v, __ddiv_rn(__dmul_rn(0.5, dt), v.w), f);
        drift(p, dt, v);
        if (WRAP)
            wrap_particle(p, i, w, im.x, im.y, im.z);
        st256(vel + i, v);
        st256(pos + i, p);
        take_particle(a, (unsigned int)i, p, c, im.x, im.y, im.z, fnew);
        }
    block_merge<true, false>(a, fnew, sc);
    if (!last_to_publish(recs, sc, ticket, s_last))
        return;
    BussiIn bz = {};
    combine_phase<true, false, false, true>(recs, (int)gridDim.x, 0ull, fnew, bz, sc, scalars, true);
    if (threadIdx.x == 0)
        {
        *fin_out = sc.fin;
        *ticket = 0ull;
        }
    }

// ONE launch per MD step (SURVEY.md 8f.1 + 8f.2 taken to the end): the second half kick of the previous step, the
// Bussi thermostat, the first half kick and the drift of this step and the dipole reduce of the new positions,
//     v1 = v + dt/2 f/m            (f = f_other + rank-1 cavity force of the previous Final record)
//     KE = 1/2 sum_group m |v1|^2  -> alpha (compute_rescale_factor, reservoir bookkeeping)
//     v2 = alpha v1 + dt/2 f/m ;  r += dt v2 ;  d += charge (r + image L)
// i.e. cavb200_nvt_step_two_rank1 of step t-1 followed by cavb200_md_step_one of step t, with every array moved
// once: vel 32 + 32, pos 32 + 32, charge 8, image 12 = 148 B/particle (the velocities are read again for the second
// pass, an L2 hit at 1M particles).  Structure of k_split_folder: 295 streaming CTAs, one folder CTA.
//     streaming CTA:  pass 1 (v1 on the fly, KE) -> publish | take alpha | pass 2 (v2, r, dipole) -> publish
//     folder CTA:     fold KE records -> alpha -> Final(K) | fold dipole records -> Scalars, Final for the next step
template<int LB, int U2, bool WRAP, bool MASK>
__global__ void __launch_bounds__(LB, LB == 384 ? 2 : 1)
    k_md_fused(double4* pos, double4* vel, const double4* force_other, uint32_t N, double dt, BussiIn b, Rank1In r1,
               ForceIn fnew, Partial* recsF, Partial* recsB, Partial* finals, Scalars* scalars,
               unsigned long long* epoch_ctr, Final* fin_out, WrapIn w, const uint32_t* mask)
    {
    __shared__ BlockScratch sc;
    __shared__ Final s_fin;
    pdl_wait();
    if (threadIdx.x == 0)
        {
        sc.flags = 0u;
        sc.epoch = ld_relaxed_u64(epoch_ctr) + 1ull;
        s_fin = *r1.fin;
        }
    __syncthreads();
    const unsigned long long epoch = sc.epoch;
    StreamGrid g;
    g.nblk = gridDim.x - 1;
    g.blk = blockIdx.x - 1;
    if (blockIdx.x == 0)
        {
        // ---- folder ----
        // Both folds are on the critical path here and their code is cold every launch: run the same loop body over
        // dummy records first (the folder has all of pass 1 to spare), then over the real ones (see k_split_folder).
        const unsigned long long dummy_epoch = ~epoch;
        Partial* dummy = recsF + MAX_PARTIALS / 4;
        for (int j = threadIdx.x; j < (int)g.nblk; j += blockDim.x)
            {
            Partial z = {};
            z.first_L = j == 0 ? 0ull : ~0ull;
            z.ke = 1.0;
            publish_record(dummy + j, z, dummy_epoch);
            }
        __syncthreads();
        bool timeout_k = false;
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++)
            {
            const bool real = pass == 1;
            const unsigned long long ep = real ? epoch : dummy_epoch;
            combine_phase<false, true, true, true, false, true>(real ? recsB : dummy, (int)g.nblk, ep, fnew, b, sc, scalars, real);
            timeout_k = sc.fin.timeout != 0;
            if (threadIdx.x == 0)
                publish_final<false>(real ? finals + 1 : dummy + g.nblk, sc.fin, ep);
            __syncthreads();
            combine_phase<true, false, true, true, false, true>(real ? recsF : dummy, (int)g.nblk, ep, fnew, b, sc, scalars, real);
            if (threadIdx.x == 0 && real)
                {
                if (timeout_k)
                    sc.fin.timeout = 1;
                *fin_out = sc.fin; // Dq, F_L, photon index of the NEW positions: the next launch's kicks use it
                *epoch_ctr = epoch;
                }
            __syncthreads();
            }
        pdl_launch_dependents();
        return;
        }
    // ---- streaming CTAs ----
    const unsigned long long stride = (unsigned long long)g.nblk * blockDim.x;
    const unsigned long long i0 = (unsigned long long)g.blk * blockDim.x + threadIdx.x;
    const unsigned long long lo = b.first, hi = (unsigned long long)b.first + b.n;
    const double half_dt = __dmul_rn(0.5, dt);
    // pass 1: kinetic energy of v1 = v + dt/2 f/m, nothing written
        {
        Acc a;
        acc_zero(a);
        double ke0 = 0.0, ke1 = 0.0;
        unsigned long long i = i0;
        for (; i + stride < N; i += 2 * stride)
            {
            const double4 va = ld256_na(vel + i), vb = ld256_na(vel + i + stride);
            const double ca = __ldg(r1.charge + i), cb = __ldg(r1.charge + i + stride);
            double4 fa = force_of(i, ca, s_fin, r1.f), fb = force_of(i + stride, cb, s_fin, r1.f);
            if (force_other)
                {
                const double4 oa = ld256(force_other + i), ob = ld256(force_other + i + stride);
                add_other(fa, oa);
                add_other(fb, ob);
                }
            const double ha = __ddiv_rn(half_dt, va.w), hb = __ddiv_rn(half_dt, vb.w);
            double4 a1 = va, b1 = vb;
            half_kick(a1, ha, fa);
            half_kick(b1, hb, fb);
            if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
                ke0 += va.w * (a1.x * a1.x + a1.y * a1.y + a1.z * a1.z);
            if (MASK ? in_mask(mask, i + stride) : i + stride >= lo && i + stride < hi)
                ke1 += vb.w * (b1.x * b1.x + b1.y * b1.y + b1.z * b1.z);
            }
        for (; i < N; i += stride)
            {
            const double4 va = ld256_na(vel + i);
            double4 fa = force_of(i, __ldg(r1.charge + i), s_fin, r1.f);
            if (force_other)
                add_other(fa, ld256(force_other + i));
            double4 a1 = va;
            half_kick(a1, __ddiv_rn(half_dt, va.w), fa);
            if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
                ke0 += va.w * (a1.x * a1.x + a1.y * a1.y + a1.z * a1.z);
            }
        a.ke = ke0 + ke1;
        block_merge<false, true>(a, fnew, sc);
        }
    if (threadIdx.x == 0)
        publish_record(recsB + g.blk, sc.rec, epoch);
    // (pulling this thread's pass-2 positions and images into L2 with prefetch.global.L2 while alpha is awaited was
    // measured: no gain at 1M, 130.4 -> 133.9 us at 4M where it evicts the velocities; not done)
    // (polling with 16 ns instead of 300 ns sleeps was measured here too: 35.92 vs 35.76 us, no better)
    const Final finK = take_final<false>(finals + 1, epoch, prefetch_final<false>(finals + 1));
    if (finK.timeout)
        {
        if (threadIdx.x == 0)
            raise_fault(scalars);
        return;
        }
    const double alpha = (b.rescale && finK.bussi_ok) ? finK.alpha : 1.0;
    // pass 2: v2 = alpha v1 + dt/2 f/m, r += dt v2, dipole term of the new position (U2 particles in flight per thread)
    Acc a;
    acc_zero(a);
    auto finish = [&](unsigned long long i, double4 v, double4 p, double c, int3 im, double4 f)
        {
        const double hm = __ddiv_rn(half_dt, v.w);
        half_kick(v, hm, f);
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            {
            v.x = __dmul_rn(v.x, alpha);
            v.y = __dmul_rn(v.y, alpha);
            v.z = __dmul_rn(v.z, alpha);
            }
        half_kick(v, hm, f);
        drift(p, dt, v);
        if (WRAP)
            wrap_particle(p, i, w, im.x, im.y, im.z);
        st256(vel + i, v);
        st256(pos + i, p);
        take_particle(a, (unsigned int)i, p, c, im.x, im.y, im.z, fnew);
        };
    unsigned long long i = i0;
    for (; i + (U2 - 1) * stride < N; i += U2 * stride)
        {
        double4 v[U2], p[U2], f[U2];
        double c[U2];
        int3 im[U2];
#pragma unroll
        for (int k = 0; k < U2; k++)
            {
            const unsigned long long j = i + k * stride;
            v[k] = ld256(vel + j);
            p[k] = ld256_na(pos + j); // coherent: this kernel overwrites pos (no .nc)
            c[k] = __ldg(r1.charge + j);
            im[k] = load_image<WRAP>(w, fnew.image, j);
            if (force_other)
                f[k] = ld256(force_other + j);
            }
#pragma unroll
        for (int k = 0; k < U2; k++)
            {
            const unsigned long long j = i + k * stride;
            double4 fc = force_of(j, c[k], s_fin, r1.f);
            if (force_other)
                add_other(fc, f[k]);
            finish(j, v[k], p[k], c[k], im[k], fc);
            }
        }
    for (; i < N; i += stride)
        {
        const double c = __ldg(r1.charge + i);
        const double4 fc = rank1_force(force_other, i, c, r1, s_fin);
        finish(i, ld256(vel + i), ld256_na(pos + i), c, load_image<WRAP>(w, fnew.image, i), fc);
        }
    block_merge<true, false>(a, fnew, sc);
    if (threadIdx.x == 0)
        publish_record(recsF + g.blk, sc.rec, epoch);
    pdl_launch_dependents();
    }

template<bool DRIFT, bool WRAP>
__global__ void __launch_bounds__(256) k_nve(double4* pos, double4* vel, const double4* force, uint32_t N, double dt, WrapIn w)
    {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        {
        double4 v = ld256(vel + i);
        const double4 f = ld256(force + i);
        half_kick(v, __ddiv_rn(__dmul_rn(0.5, dt), v.w), f);
        st256(vel + i, v);
        if (DRIFT)
            {
            double4 p = ld256(pos + i);
            drift(p, dt, v);
            if (WRAP)
                {
                int ix = w.image[3 * i + 0], iy = w.image[3 * i + 1], iz = w.image[3 * i + 2];
                wrap_particle(p, i, w, ix, iy, iz);
                }
            st256(pos + i, p);
            }
        }
    }

// Group mask from an index list (the words were zeroed before the launch): bit idx[k] of the mask is set.  bad gets
// bit 0 for an index >= N and bit 1 for an index that is listed twice (its bit was already set).
__global__ void __launch_bounds__(256) k_group_mask(const uint32_t* idx, uint32_t n, uint32_t N, uint32_t* mask,
                                                    unsigned long long* bad)
    {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
        {
        const uint32_t i = __ldg(idx + k);
        if (i >= N)
            {
            atomicOr(bad, 1ull);
            continue;
            }
        const uint32_t bit = 1u << (i & 31);
        if (atomicOr(mask + (i >> 5), bit) & bit)
            atomicOr(bad, 2ull);
        }
    }

// After the particle arrays were permuted: the lowest index whose type id (low 32 bits of pos.w) is L_typeid, and how
// many such particles there are, in s[0] / s[1] (set to ~0 / 0 before the launch).  The last CTA to take the ticket
// s[2] patches the rank-1 Final record when there is exactly one: photon_local is the only field of it that depends on
// the order of the particles (Dq, F_L and the energies are sums and products over the whole system).
__global__ void __launch_bounds__(256) k_photon_reindex(const double4* pos, uint32_t N, uint32_t L_typeid,
                                                        unsigned long long* s, Final* fin)
    {
    unsigned int first = NO_INDEX, cnt = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        if (__double2loint(__ldg(&pos[i].w)) == (int)L_typeid)
            {
            first = first < (unsigned int)i ? first : (unsigned int)i;
            cnt++;
            }
    first = __reduce_min_sync(0xffffffffu, first);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt)
        {
        atomicMin(s, (unsigned long long)first);
        atomicAdd(s + 1, (unsigned long long)cnt);
        }
    __syncthreads();
    if (threadIdx.x == 0)
        {
        __threadfence();
        const bool last = atom_acq_rel_add_u64(s + 2, 1ull) == (unsigned long long)gridDim.x - 1;
        if (last && ld_relaxed_u64(s + 1) == 1ull)
            {
            fin->photon_local = (long long)ld_relaxed_u64(s);
            fin->many_L = 0;
            }
        }
    }
    } // namespace cavb

using namespace cavb;

// net_force[i] += cavity force of particle i, formed from the charge (SURVEY.md 8f.2): what a net-force
// summing kernel does with the rank-1 contribution instead of reading a stored force array
__global__ void __launch_bounds__(256) k_net_force_add_rank1(double4* net, uint32_t N, Rank1In r1)
    {
    __shared__ Final s_fin;
    if (threadIdx.x == 0)
        s_fin = *r1.fin;
    __syncthreads();
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride)
        st256(net + i, kick_force<true>(net, i, r1, s_fin));
    }

// f(std::bool_constant<b0>{}, std::bool_constant<b1>{}, ...): one launch statement instantiates a kernel for every
// combination of its bool template parameters and launches the one the run-time flags select
template<class F>
static void with_flags(F&& f)
    {
    f();
    }
template<class F, class... B>
static void with_flags(F&& f, bool b0, B... rest)
    {
    if (b0)
        with_flags([&](auto... t) { f(std::true_type{}, t...); }, rest...);
    else
        with_flags([&](auto... t) { f(std::false_type{}, t...); }, rest...);
    }

// Grid of a grid-stride launch of 256-thread CTAs over n items: one CTA per 256 items, at most ctas_per_sm CTAs per SM
// and, for a kernel that leaves one record per CTA in the partials bank, at most MAX_PARTIALS.  The grid size also sets
// the order in which those records are folded, i.e. the bits of the sums.
static int grid_for(const cavb200_handle* h, unsigned long long n, int ctas_per_sm, bool cap_partials = false)
    {
    unsigned long long cap = (unsigned long long)h->num_sms * ctas_per_sm;
    if (cap_partials && cap > (unsigned long long)MAX_PARTIALS)
        cap = MAX_PARTIALS;
    const unsigned long long want = (n + 255) / 256;
    return (int)(want < cap ? want : cap);
    }

// after a <<<...>>> launch: its error, or count it
static int launched(cavb200_handle* h)
    {
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

// The thermostatted group of the window entry points: [group_first, group_first + n_group), or, with group_first ==
// CAVB200_GROUP_MASK, the mask of the last cavb200_group_set (which must have been made for n_group members of N
// particles).  Returns false for a group that does not fit; *mask is the mask to pass to the kernels, or NULL.
static bool group_ok(const cavb200_handle* h, uint32_t N, uint32_t group_first, uint32_t n_group, const uint32_t** mask)
    {
    *mask = nullptr;
    if (group_first != CAVB200_GROUP_MASK)
        return (unsigned long long)group_first + n_group <= N;
    if (!h->group_ready || n_group != h->group_n || N != h->group_N)
        return false;
    *mask = h->group_mask;
    return true;
    }

// The thermostat arguments of the harness kernels: the group and, with bussi given and deltaT != 0, the rescale
static BussiIn harness_bussi(uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi)
    {
    BussiIn b = {};
    b.first = group_first;
    b.n = n_group;
    b.rescale = bussi != nullptr && bussi->deltaT != 0.0;
    if (bussi)
        fill_bussi_constants(b, bussi);
    return b;
    }

// The rank-1 arguments of an entry point as the kernels take them.  h may still be NULL here; the launcher rejects that
// before it looks at anything else.
static Rank1In rank1_in(const cavb200_handle* h, const double* charge, const double* pos, uint32_t L_typeid, double couplstr)
    {
    Rank1In r = Rank1In();
    r.charge = charge;
    r.fin = h ? rank1_final(h) : nullptr;
    r.f.pos = reinterpret_cast<const double4*>(pos);
    r.f.L_typeid = L_typeid;
    r.f.g = couplstr;
    return r;
    }

// Checks of the rank-1 and box-wrap arguments of a call (NULL: the call has none)
static int check_rank1_wrap(const Rank1In* r1, const WrapIn* w)
    {
    if ((r1 && (!r1->charge || !r1->f.pos)) || (w && (!w->image || !(w->Lx > 0.0) || !(w->Ly > 0.0) || !(w->Lz > 0.0))))
        return (int)cudaErrorInvalidValue;
    if ((r1 && (misaligned(r1->f.pos, 32) || misaligned(r1->charge, 8))) || (w && misaligned(w->image, 4)))
        return (int)cudaErrorMisalignedAddress;
    return 0;
    }

static int nve_launch(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt, void* stream,
                      bool drift, const WrapIn* w = nullptr)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    if (!vel || !force || (drift && !pos))
        return (int)cudaErrorInvalidValue;
    if (misaligned(pos, 32) || misaligned(vel, 32) || misaligned(force, 32))
        return (int)cudaErrorMisalignedAddress;
    if (const int rc = check_rank1_wrap(nullptr, w))
        return rc;
    const WrapIn wr = w ? *w : WrapIn();
    const int grid = grid_for(h, N, 8);
    with_flags(
        [&](auto DRIFT, auto WRAP)
        {
            if constexpr (DRIFT || !WRAP) // (the wrap comes with the drift only)
                k_nve<DRIFT, WRAP><<<grid, 256, 0, (cudaStream_t)stream>>>((double4*)pos, (double4*)vel,
                                                                          (const double4*)force, N, dt, wr);
        },
        drift, w != nullptr);
    return launched(h);
    }

static int nvt_one(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                   uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream,
                   const Rank1In* r1 = nullptr, const WrapIn* w = nullptr)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    if (const int rc = check_rank1_wrap(r1, w))
        return rc;
    const uint32_t* mask;
    if (!pos || !vel || (!force && !r1) || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (misaligned(pos, 32) || misaligned(vel, 32) || misaligned(force, 32))
        return (int)cudaErrorMisalignedAddress;
    const BussiIn b = harness_bussi(group_first, n_group, bussi);
    const Rank1In r = r1 ? *r1 : Rank1In();
    const WrapIn wr = w ? *w : WrapIn();
    const int grid = grid_for(h, N, CAVB_NVT_CTAS_PER_SM);
    with_flags(
        [&](auto RANK1, auto WRAP, auto MASK)
        {
            k_nvt_one<RANK1, WRAP, MASK><<<grid, 256, 0, (cudaStream_t)stream>>>(
                (double4*)pos, (double4*)vel, (const double4*)force, N, dt, b, h->scalars, r, wr, mask);
        },
        r1 != nullptr, w != nullptr, mask != nullptr);
    return launched(h);
    }

static int nvt_two(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt, uint32_t group_first,
                   uint32_t n_group, void* stream, const Rank1In* r1 = nullptr)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    if (const int rc = check_rank1_wrap(r1, nullptr))
        return rc;
    const uint32_t* mask;
    if (!vel || (!force && !r1) || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (misaligned(vel, 32) || misaligned(force, 32))
        return (int)cudaErrorMisalignedAddress;
    const BussiIn b = harness_bussi(group_first, n_group, nullptr);
    const Rank1In r = r1 ? *r1 : Rank1In();
    const int grid = grid_for(h, N, CAVB_NVT_CTAS_PER_SM, true);
    with_flags(
        [&](auto RANK1, auto MASK)
        {
            k_nvt_two<RANK1, MASK><<<grid, 256, 0, (cudaStream_t)stream>>>((double4*)vel, (const double4*)force, N, dt, b,
                                                                          h->partials, h->scalars, h->counters + 4, r, mask);
        },
        r1 != nullptr, mask != nullptr);
    return launched(h);
    }

extern "C" int cavb200_nve_kick_drift(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N,
                                      double dt, void* stream)
    {
    return nve_launch(h, pos, vel, force, N, dt, stream, true);
    }

extern "C" int cavb200_nve_kick_drift_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image,
                                           uint32_t N, double dt, double Lx, double Ly, double Lz, void* stream)
    {
    const WrapIn w = {image, Lx, Ly, Lz};
    return nve_launch(h, pos, vel, force, N, dt, stream, true, &w);
    }

extern "C" int cavb200_nve_half_kick(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt,
                                     void* stream)
    {
    return nve_launch(h, nullptr, vel, force, N, dt, stream, false);
    }

extern "C" int cavb200_nvt_step_one(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                                    uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    return nvt_one(h, pos, vel, force, N, dt, group_first, n_group, bussi, stream);
    }

extern "C" int cavb200_nvt_step_one_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image,
                                         uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t group_first,
                                         uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    const WrapIn w = {image, Lx, Ly, Lz};
    return nvt_one(h, pos, vel, force, N, dt, group_first, n_group, bussi, stream, nullptr, &w);
    }

extern "C" int cavb200_nvt_step_two(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt,
                                    uint32_t group_first, uint32_t n_group, void* stream)
    {
    return nvt_two(h, vel, force, N, dt, group_first, n_group, stream);
    }

extern "C" int cavb200_nvt_step_one_rank1(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                          const double* charge, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                                          uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                                          void* stream)
    {
    const Rank1In r = rank1_in(h, charge, pos, L_typeid, couplstr);
    return nvt_one(h, pos, vel, force_other, N, dt, group_first, n_group, bussi, stream, &r);
    }

extern "C" int cavb200_nvt_step_one_rank1_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                               const double* charge, int32_t* image, uint32_t N, double dt, double Lx,
                                               double Ly, double Lz, uint32_t L_typeid, double couplstr,
                                               uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                                               void* stream)
    {
    const Rank1In r = rank1_in(h, charge, pos, L_typeid, couplstr);
    const WrapIn w = {image, Lx, Ly, Lz};
    return nvt_one(h, pos, vel, force_other, N, dt, group_first, n_group, bussi, stream, &r, &w);
    }

extern "C" int cavb200_nvt_step_two_rank1(cavb200_handle* h, double* vel, const double* force_other, const double* charge,
                                          const double* pos, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                                          uint32_t group_first, uint32_t n_group, void* stream)
    {
    const Rank1In r = rank1_in(h, charge, pos, L_typeid, couplstr);
    return nvt_two(h, vel, force_other, N, dt, group_first, n_group, stream, &r);
    }

// The arguments of k_md_one and k_md_fused
struct MdArgs
    {
    const uint32_t* mask;
    BussiIn b;
    Rank1In r;
    ForceIn fnew;
    WrapIn w;
    };

static int md_args(MdArgs& a, cavb200_handle* h, const double* pos, const double* vel, const double* force_other,
                   const double* charge, const int32_t* image, uint32_t N, double Lx, double Ly, double Lz,
                   uint32_t L_typeid, const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                   const cavb200_bussi_args* bussi, bool wrap)
    {
    if (!vel || !group_ok(h, N, group_first, n_group, &a.mask))
        return (int)cudaErrorInvalidValue;
    if (misaligned(vel, 32) || misaligned(force_other, 32))
        return (int)cudaErrorMisalignedAddress;
    a.fnew = ForceIn();
    if (const int rc = fill_force(a.fnew, pos, charge, image, nullptr, N, Lx, Ly, Lz, L_typeid, params, 0, false))
        return rc;
    a.b = harness_bussi(group_first, n_group, bussi);
    a.r = rank1_in(h, charge, pos, L_typeid, params->couplstr);
    a.w = wrap ? WrapIn{const_cast<int32_t*>(image), Lx, Ly, Lz} : WrapIn();
    return check_rank1_wrap(nullptr, wrap ? &a.w : nullptr);
    }

static int md_step_one_impl(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                            const double* charge, const int32_t* image, uint32_t N, double dt, double Lx, double Ly,
                            double Lz, uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                            uint32_t n_group, const cavb200_bussi_args* bussi, void* stream, bool wrap)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    MdArgs a;
    if (const int rc = md_args(a, h, pos, vel, force_other, charge, image, N, Lx, Ly, Lz, L_typeid, params, group_first,
                               n_group, bussi, wrap))
        return rc;
    const int grid = grid_for(h, N, 3, true); // one wave of 3 CTAs per SM (85-register budget)
    Final* fin_out = const_cast<Final*>(rank1_final(h));
    with_flags(
        [&](auto WRAP, auto MASK)
        {
            k_md_one<WRAP, MASK><<<grid, 256, 0, (cudaStream_t)stream>>>((double4*)pos, (double4*)vel,
                                                                        (const double4*)force_other, N, dt, a.b, h->scalars,
                                                                        a.r, a.fnew, h->partials, h->counters + 4, fin_out,
                                                                        a.w, a.mask);
        },
        wrap, a.mask != nullptr);
    return launched(h);
    }

extern "C" int cavb200_md_step_one(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                   const double* charge, const int32_t* image, uint32_t N, double dt, double Lx, double Ly,
                                   double Lz, uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                                   uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    return md_step_one_impl(h, pos, vel, force_other, charge, image, N, dt, Lx, Ly, Lz, L_typeid, params, group_first, n_group,
                            bussi, stream, false);
    }

extern "C" int cavb200_md_step_one_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                        const double* charge, int32_t* image, uint32_t N, double dt, double Lx, double Ly,
                                        double Lz, uint32_t L_typeid, const cavb200_params* params, uint32_t group_first,
                                        uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    return md_step_one_impl(h, pos, vel, force_other, charge, image, N, dt, Lx, Ly, Lz, L_typeid, params, group_first, n_group,
                            bussi, stream, true);
    }

static int md_step_fused_impl(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                              const double* charge, const int32_t* image, uint32_t N, double dt, double Lx,
                              double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params,
                              uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream, bool wrap)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    MdArgs a;
    if (const int rc = md_args(a, h, pos, vel, force_other, charge, image, N, Lx, Ly, Lz, L_typeid, params, group_first,
                               n_group, bussi, wrap))
        return rc;
    if (!h->coop_supported)
        return (int)cudaErrorNotSupported;
    if (const int fault = check_fault(h))
        return fault;
    // md_shape 1: two 384-thread CTAs per SM; otherwise one 768-thread CTA per SM (the folder CTA alone on its SM)
    const bool two = h->tune.md_shape == 1;
    const int threads = two ? 384 : 768, per_sm_want = two ? 2 : 1;
    const void* kern;
    with_flags([&](auto TWO, auto WRAP, auto MASK) { kern = (const void*)k_md_fused<TWO ? 384 : 768, 1, WRAP, MASK>; },
               two, wrap, a.mask != nullptr);
    int per_sm = 0;
    CAVB_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, 0));
    if (per_sm < 1)
        return (int)cudaErrorLaunchOutOfResources;
    if (per_sm > per_sm_want)
        per_sm = per_sm_want;
    int max_grid = per_sm * h->num_sms;
    if (max_grid > MAX_PARTIALS / 4 - 2)
        max_grid = MAX_PARTIALS / 4 - 2;
    const unsigned long long want = ((unsigned long long)N + threads - 1) / threads;
    // the CTAs wait on each other: the grid must be co-resident; one of them folds instead of streaming
    const int grid = (int)(want < (unsigned long long)(max_grid - 1) ? want : (unsigned long long)(max_grid - 1)) + 1;
    double4* p4 = (double4*)pos;
    double4* v4 = (double4*)vel;
    const double4* fo4 = (const double4*)force_other;
    Partial* recsF = h->partials;
    Partial* recsB = h->partials + MAX_PARTIALS / 2;
    Partial* finals = h->partials + MAX_PARTIALS - 2;
    Scalars* sca = h->scalars;
    unsigned long long* ctr = h->counters + 2;
    Final* fin_out = const_cast<Final*>(rank1_final(h));
    void* args[] = {&p4, &v4, &fo4, &N, &dt, &a.b, &a.r, &a.fnew, &recsF, &recsB, &finals, &sca, &ctr, &fin_out, &a.w, &a.mask};
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr;
    if (h->tune.pdl)
        {
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        }
    else
        {
        attr.id = cudaLaunchAttributeCooperative;
        attr.val.cooperative = 1;
        }
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    CAVB_CHECK(cudaLaunchKernelExC(&cfg, kern, args));
    h->launches += 1;
    return 0;
    }

extern "C" int cavb200_md_step_fused(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                     const double* charge, const int32_t* image, uint32_t N, double dt, double Lx,
                                     double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params,
                                     uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    return md_step_fused_impl(h, pos, vel, force_other, charge, image, N, dt, Lx, Ly, Lz, L_typeid, params, group_first,
                              n_group, bussi, stream, false);
    }

extern "C" int cavb200_md_step_fused_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                          const double* charge, int32_t* image, uint32_t N, double dt, double Lx,
                                          double Ly, double Lz, uint32_t L_typeid, const cavb200_params* params,
                                          uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                                          void* stream)
    {
    return md_step_fused_impl(h, pos, vel, force_other, charge, image, N, dt, Lx, Ly, Lz, L_typeid, params, group_first,
                              n_group, bussi, stream, true);
    }

extern "C" int cavb200_net_force_add_rank1(cavb200_handle* h, double* net_force, const double* charge, const double* pos,
                                           uint32_t N, uint32_t L_typeid, double couplstr, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    if (!net_force)
        return (int)cudaErrorInvalidValue;
    if (misaligned(net_force, 32))
        return (int)cudaErrorMisalignedAddress;
    const Rank1In r = rank1_in(h, charge, pos, L_typeid, couplstr);
    if (const int rc = check_rank1_wrap(&r, nullptr))
        return rc;
    k_net_force_add_rank1<<<grid_for(h, N, 8), 256, 0, (cudaStream_t)stream>>>((double4*)net_force, N, r);
    return launched(h);
    }

// ---- index-list groups ---------------------------------------------------------------------------------------------
extern "C" int cavb200_group_set(cavb200_handle* h, const uint32_t* group_idx, uint32_t n, uint32_t N, void* stream)
    {
    if (!h || (n && !group_idx))
        return (int)cudaErrorInvalidValue;
    if (reinterpret_cast<uintptr_t>(group_idx) & 3)
        return (int)cudaErrorMisalignedAddress;
    h->group_ready = 0;
    const unsigned long long words = ((unsigned long long)N + 31) / 32;
    if (words > h->group_mask_words)
        {
        cudaFree(h->group_mask);
        h->group_mask = nullptr;
        h->group_mask_words = 0;
        CAVB_CHECK(cudaMalloc((void**)&h->group_mask, words * sizeof(uint32_t)));
        h->group_mask_words = words;
        }
    cudaStream_t cs = (cudaStream_t)stream;
    unsigned long long* bad = h->counters + 48;
    CAVB_CHECK(cudaMemsetAsync(bad, 0, sizeof(unsigned long long), cs));
    if (words)
        CAVB_CHECK(cudaMemsetAsync(h->group_mask, 0, words * sizeof(uint32_t), cs));
    if (n)
        {
        k_group_mask<<<grid_for(h, n, 8), 256, 0, cs>>>(group_idx, n, N, h->group_mask, bad);
        CAVB_CHECK(cudaGetLastError());
        h->launches += 1;
        }
    unsigned long long flags = 0;
    CAVB_CHECK(cudaMemcpyAsync(&flags, bad, sizeof(flags), cudaMemcpyDeviceToHost, cs));
    CAVB_CHECK(cudaStreamSynchronize(cs));
    if (flags)
        return (int)cudaErrorInvalidValue; // an index >= N (bit 0) or one listed twice (bit 1)
    h->group_n = n;
    h->group_N = N;
    h->group_ready = 1;
    return 0;
    }

extern "C" int cavb200_rank1_reindex(cavb200_handle* h, const double* pos, uint32_t N, uint32_t L_typeid, void* stream)
    {
    if (!h || (N && !pos))
        return (int)cudaErrorInvalidValue;
    if (misaligned(pos, 32))
        return (int)cudaErrorMisalignedAddress;
    if (N == 0)
        return 0;
    cudaStream_t cs = (cudaStream_t)stream;
    unsigned long long* sc = h->counters + 49; // {first, count, ticket}
    CAVB_CHECK(cudaMemsetAsync(sc, 0xFF, sizeof(unsigned long long), cs));
    CAVB_CHECK(cudaMemsetAsync(sc + 1, 0, 2 * sizeof(unsigned long long), cs));
    k_photon_reindex<<<grid_for(h, N, 8), 256, 0, cs>>>(reinterpret_cast<const double4*>(pos), N, L_typeid, sc,
                                                        const_cast<Final*>(rank1_final(h)));
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    unsigned long long found[2];
    CAVB_CHECK(cudaMemcpyAsync(found, sc, sizeof(found), cudaMemcpyDeviceToHost, cs));
    CAVB_CHECK(cudaStreamSynchronize(cs));
    // several 'L' particles: which of them F_L was computed for is not recorded, so the first one by index after a sort
    // need not be it
    return found[1] > 1 ? (int)cudaErrorNotSupported : 0;
    }
