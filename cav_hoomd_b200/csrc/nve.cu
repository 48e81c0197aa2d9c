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

template<bool RANK1>
__device__ __forceinline__ double4 kick_force(const double4* force, unsigned long long i, const Rank1In& r, const Final& fin)
    {
    if (!RANK1)
        return ld256(force + i);
    double4 fc = force_of(i, __ldg(r.charge + i), fin, r.f);
    if (force)
        {
        const double4 fo = ld256(force + i);
        fc.x = __dadd_rn(fo.x, fc.x);
        fc.y = __dadd_rn(fo.y, fc.y);
        fc.z = __dadd_rn(fo.z, fc.z);
        fc.w = fo.w; // potential-energy slot of the other forces; the cavity term's is 0 (:145,180)
        }
    return fc;
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
        s_alpha = alpha;
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
        const double hm = __ddiv_rn(__dmul_rn(0.5, dt), v.w);
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        p.x = __dadd_rn(p.x, __dmul_rn(dt, v.x));
        p.y = __dadd_rn(p.y, __dmul_rn(dt, v.y));
        p.z = __dadd_rn(p.z, __dmul_rn(dt, v.z));
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
        const double hm = __ddiv_rn(__dmul_rn(0.5, dt), v.w);
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        st256(vel + i, v);
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            a.ke += v.w * (v.x * v.x + v.y * v.y + v.z * v.z);
        }
    ForceIn f0 = {};
    block_merge<false, true>(a, f0, sc);
    if (threadIdx.x == 0)
        {
        publish_record(recs + blockIdx.x, sc.rec, 0ull);
        __threadfence();
        const unsigned long long t = atom_acq_rel_add_u64(ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
        }
    __syncthreads();
    if (!s_last)
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
                    const double inst = __dmul_rn(KE, __dadd_rn(1.0, -__dmul_rn(alpha, alpha))); // BussiReservoirThermostat.h:86-95
                    scalars->alpha = alpha;
                    scalars->inst = inst;
                    scalars->cumulative = __dadd_rn(scalars->cumulative, inst);
                    }
                scalars->err = ok ? 0.0 : 1.0;
                }
            }
        s_alpha = alpha;
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
        // (WRAP: this kernel rewrites the image flags, so they are read coherently, not through the read-only path)
        int ix = WRAP ? w.image[3 * i + 0] : __ldg(fnew.image + 3 * i + 0);
        int iy = WRAP ? w.image[3 * i + 1] : __ldg(fnew.image + 3 * i + 1);
        int iz = WRAP ? w.image[3 * i + 2] : __ldg(fnew.image + 3 * i + 2);
        double4 f = force_of(i, c, s_fin, r1.f);
        if (force_other)
            {
            const double4 fo = ld256(force_other + i);
            f.x = __dadd_rn(fo.x, f.x);
            f.y = __dadd_rn(fo.y, f.y);
            f.z = __dadd_rn(fo.z, f.z);
            }
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            {
            v.x = __dmul_rn(v.x, alpha);
            v.y = __dmul_rn(v.y, alpha);
            v.z = __dmul_rn(v.z, alpha);
            }
        const double hm = __ddiv_rn(__dmul_rn(0.5, dt), v.w);
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        p.x = __dadd_rn(p.x, __dmul_rn(dt, v.x));
        p.y = __dadd_rn(p.y, __dmul_rn(dt, v.y));
        p.z = __dadd_rn(p.z, __dmul_rn(dt, v.z));
        if (WRAP)
            wrap_particle(p, i, w, ix, iy, iz);
        st256(vel + i, v);
        st256(pos + i, p);
        take_particle(a, (unsigned int)i, p, c, ix, iy, iz, fnew);
        }
    block_merge<true, false>(a, fnew, sc);
    if (threadIdx.x == 0)
        {
        publish_record(recs + blockIdx.x, sc.rec, 0ull);
        __threadfence();
        const unsigned long long t = atom_acq_rel_add_u64(ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
        }
    __syncthreads();
    if (!s_last)
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
                fa.x = __dadd_rn(oa.x, fa.x); fa.y = __dadd_rn(oa.y, fa.y); fa.z = __dadd_rn(oa.z, fa.z);
                fb.x = __dadd_rn(ob.x, fb.x); fb.y = __dadd_rn(ob.y, fb.y); fb.z = __dadd_rn(ob.z, fb.z);
                }
            const double ha = __ddiv_rn(half_dt, va.w), hb = __ddiv_rn(half_dt, vb.w);
            const double ax = __dadd_rn(va.x, __dmul_rn(ha, fa.x)), ay = __dadd_rn(va.y, __dmul_rn(ha, fa.y)),
                         az = __dadd_rn(va.z, __dmul_rn(ha, fa.z));
            const double bx = __dadd_rn(vb.x, __dmul_rn(hb, fb.x)), by = __dadd_rn(vb.y, __dmul_rn(hb, fb.y)),
                         bz = __dadd_rn(vb.z, __dmul_rn(hb, fb.z));
            if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
                ke0 += va.w * (ax * ax + ay * ay + az * az);
            if (MASK ? in_mask(mask, i + stride) : i + stride >= lo && i + stride < hi)
                ke1 += vb.w * (bx * bx + by * by + bz * bz);
            }
        for (; i < N; i += stride)
            {
            const double4 va = ld256_na(vel + i);
            double4 fa = force_of(i, __ldg(r1.charge + i), s_fin, r1.f);
            if (force_other)
                {
                const double4 oa = ld256(force_other + i);
                fa.x = __dadd_rn(oa.x, fa.x); fa.y = __dadd_rn(oa.y, fa.y); fa.z = __dadd_rn(oa.z, fa.z);
                }
            const double ha = __ddiv_rn(half_dt, va.w);
            const double ax = __dadd_rn(va.x, __dmul_rn(ha, fa.x)), ay = __dadd_rn(va.y, __dmul_rn(ha, fa.y)),
                         az = __dadd_rn(va.z, __dmul_rn(ha, fa.z));
            if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
                ke0 += va.w * (ax * ax + ay * ay + az * az);
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
    auto finish = [&](unsigned long long i, double4 v, double4 p, double c, int ix, int iy, int iz, double4 f)
        {
        const double hm = __ddiv_rn(half_dt, v.w);
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        if (MASK ? in_mask(mask, i) : i >= lo && i < hi)
            {
            v.x = __dmul_rn(v.x, alpha);
            v.y = __dmul_rn(v.y, alpha);
            v.z = __dmul_rn(v.z, alpha);
            }
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        p.x = __dadd_rn(p.x, __dmul_rn(dt, v.x));
        p.y = __dadd_rn(p.y, __dmul_rn(dt, v.y));
        p.z = __dadd_rn(p.z, __dmul_rn(dt, v.z));
        if (WRAP)
            wrap_particle(p, i, w, ix, iy, iz);
        st256(vel + i, v);
        st256(pos + i, p);
        take_particle(a, (unsigned int)i, p, c, ix, iy, iz, fnew);
        };
    unsigned long long i = i0;
    for (; i + (U2 - 1) * stride < N; i += U2 * stride)
        {
        double4 v[U2], p[U2], f[U2];
        double c[U2];
        int ix[U2], iy[U2], iz[U2];
#pragma unroll
        for (int k = 0; k < U2; k++)
            {
            const unsigned long long j = i + k * stride;
            v[k] = ld256(vel + j);
            p[k] = ld256_na(pos + j); // coherent: this kernel overwrites pos (no .nc)
            c[k] = __ldg(r1.charge + j);
            ix[k] = WRAP ? w.image[3 * j + 0] : __ldg(fnew.image + 3 * j + 0);
            iy[k] = WRAP ? w.image[3 * j + 1] : __ldg(fnew.image + 3 * j + 1);
            iz[k] = WRAP ? w.image[3 * j + 2] : __ldg(fnew.image + 3 * j + 2);
            if (force_other)
                f[k] = ld256(force_other + j);
            }
#pragma unroll
        for (int k = 0; k < U2; k++)
            {
            const unsigned long long j = i + k * stride;
            double4 fc = force_of(j, c[k], s_fin, r1.f);
            if (force_other)
                {
                fc.x = __dadd_rn(f[k].x, fc.x);
                fc.y = __dadd_rn(f[k].y, fc.y);
                fc.z = __dadd_rn(f[k].z, fc.z);
                }
            finish(j, v[k], p[k], c[k], ix[k], iy[k], iz[k], fc);
            }
        }
    for (; i < N; i += stride)
        {
        const double c = __ldg(r1.charge + i);
        double4 fc = force_of(i, c, s_fin, r1.f);
        if (force_other)
            {
            const double4 fo = ld256(force_other + i);
            fc.x = __dadd_rn(fo.x, fc.x);
            fc.y = __dadd_rn(fo.y, fc.y);
            fc.z = __dadd_rn(fo.z, fc.z);
            }
        finish(i, ld256(vel + i), ld256_na(pos + i), c, WRAP ? w.image[3 * i + 0] : __ldg(fnew.image + 3 * i + 0),
               WRAP ? w.image[3 * i + 1] : __ldg(fnew.image + 3 * i + 1),
               WRAP ? w.image[3 * i + 2] : __ldg(fnew.image + 3 * i + 2), fc);
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
        const double hm = __ddiv_rn(__dmul_rn(0.5, dt), v.w);
        v.x = __dadd_rn(v.x, __dmul_rn(hm, f.x));
        v.y = __dadd_rn(v.y, __dmul_rn(hm, f.y));
        v.z = __dadd_rn(v.z, __dmul_rn(hm, f.z));
        st256(vel + i, v);
        if (DRIFT)
            {
            double4 p = ld256(pos + i);
            p.x = __dadd_rn(p.x, __dmul_rn(dt, v.x));
            p.y = __dadd_rn(p.y, __dmul_rn(dt, v.y));
            p.z = __dadd_rn(p.z, __dmul_rn(dt, v.z));
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

static int make_wrap(WrapIn& w, int32_t* image, double Lx, double Ly, double Lz)
    {
    if (!image || !(Lx > 0.0) || !(Ly > 0.0) || !(Lz > 0.0))
        return (int)cudaErrorInvalidValue;
    if (reinterpret_cast<uintptr_t>(image) & 3)
        return (int)cudaErrorMisalignedAddress;
    w.image = image;
    w.Lx = Lx;
    w.Ly = Ly;
    w.Lz = Lz;
    return 0;
    }

static int nve_launch(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                      cudaStream_t s, bool drift, const WrapIn* w = nullptr)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    if (!vel || !force || (drift && !pos))
        return (int)cudaErrorInvalidValue;
    if ((reinterpret_cast<uintptr_t>(pos) | reinterpret_cast<uintptr_t>(vel) | reinterpret_cast<uintptr_t>(force)) & 31)
        return (int)cudaErrorMisalignedAddress;
    unsigned long long want = ((unsigned long long)N + 255) / 256;
    const unsigned long long cap = (unsigned long long)h->num_sms * 8;
    const int grid = (int)(want < cap ? want : cap);
    if (drift && w)
        k_nve<true, true><<<grid, 256, 0, s>>>((double4*)pos, (double4*)vel, (const double4*)force, N, dt, *w);
    else if (drift)
        k_nve<true, false><<<grid, 256, 0, s>>>((double4*)pos, (double4*)vel, (const double4*)force, N, dt, WrapIn());
    else
        k_nve<false, false><<<grid, 256, 0, s>>>(nullptr, (double4*)vel, (const double4*)force, N, dt, WrapIn());
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

extern "C" int cavb200_nve_kick_drift(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N,
                                      double dt, void* stream)
    {
    return nve_launch(h, pos, vel, force, N, dt, (cudaStream_t)stream, true);
    }

extern "C" int cavb200_nve_kick_drift_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image,
                                           uint32_t N, double dt, double Lx, double Ly, double Lz, void* stream)
    {
    WrapIn w;
    if (const int rc = make_wrap(w, image, Lx, Ly, Lz))
        return rc;
    return nve_launch(h, pos, vel, force, N, dt, (cudaStream_t)stream, true, &w);
    }

extern "C" int cavb200_nve_half_kick(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt,
                                     void* stream)
    {
    return nve_launch(h, nullptr, vel, force, N, dt, (cudaStream_t)stream, false);
    }

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

static bool mis32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31) != 0; }

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

static int fill_rank1(cavb200_handle* h, Rank1In& r, const double* charge, const double* pos, uint32_t L_typeid,
                      double couplstr)
    {
    if (!charge || !pos)
        return (int)cudaErrorInvalidValue;
    if (mis32(pos) || (reinterpret_cast<uintptr_t>(charge) & 7))
        return (int)cudaErrorMisalignedAddress;
    r = Rank1In();
    r.charge = charge;
    r.fin = rank1_final(h);
    r.f.pos = reinterpret_cast<const double4*>(pos);
    r.f.L_typeid = L_typeid;
    r.f.g = couplstr;
    return 0;
    }

static int nvt_one(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                   uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, const Rank1In* r1, void* stream,
                   const WrapIn* w = nullptr)
    {
    const uint32_t* mask;
    if (!pos || !vel || (!force && !r1) || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (mis32(pos) || mis32(vel) || mis32(force))
        return (int)cudaErrorMisalignedAddress;
    BussiIn b = {};
    b.first = group_first;
    b.n = n_group;
    b.rescale = bussi != nullptr && bussi->deltaT != 0.0;
    if (bussi)
        fill_bussi_constants(b, bussi);
    unsigned long long want = ((unsigned long long)N + 255) / 256;
    const unsigned long long cap = (unsigned long long)h->num_sms * CAVB_NVT_CTAS_PER_SM;
    const int grid = (int)(want < cap ? want : cap);
    cudaStream_t cs = (cudaStream_t)stream;
    double4 *p4 = (double4*)pos, *v4 = (double4*)vel;
    const double4* f4 = (const double4*)force;
    const Rank1In r = r1 ? *r1 : Rank1In();
    const WrapIn wr = w ? *w : WrapIn();
    if (mask)
        {
        if (r1 && w)
            k_nvt_one<true, true, true><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, mask);
        else if (r1)
            k_nvt_one<true, false, true><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, mask);
        else if (w)
            k_nvt_one<false, true, true><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, mask);
        else
            k_nvt_one<false, false, true><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, mask);
        }
    else if (r1 && w)
        k_nvt_one<true, true, false><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, nullptr);
    else if (r1)
        k_nvt_one<true, false, false><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, nullptr);
    else if (w)
        k_nvt_one<false, true, false><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, nullptr);
    else
        k_nvt_one<false, false, false><<<grid, 256, 0, cs>>>(p4, v4, f4, N, dt, b, h->scalars, r, wr, nullptr);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

static int nvt_two(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt, uint32_t group_first,
                   uint32_t n_group, const Rank1In* r1, void* stream)
    {
    const uint32_t* mask;
    if (!vel || (!force && !r1) || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (mis32(vel) || mis32(force))
        return (int)cudaErrorMisalignedAddress;
    BussiIn b = {};
    b.first = group_first;
    b.n = n_group;
    unsigned long long want = ((unsigned long long)N + 255) / 256;
    unsigned long long cap = (unsigned long long)h->num_sms * CAVB_NVT_CTAS_PER_SM;
    if (cap > (unsigned long long)MAX_PARTIALS)
        cap = MAX_PARTIALS;
    const int grid = (int)(want < cap ? want : cap);
    cudaStream_t cs = (cudaStream_t)stream;
    double4* v4 = (double4*)vel;
    const double4* f4 = (const double4*)force;
    const Rank1In r = r1 ? *r1 : Rank1In();
    if (r1 && mask)
        k_nvt_two<true, true><<<grid, 256, 0, cs>>>(v4, f4, N, dt, b, h->partials, h->scalars, h->counters + 4, r, mask);
    else if (r1)
        k_nvt_two<true, false><<<grid, 256, 0, cs>>>(v4, f4, N, dt, b, h->partials, h->scalars, h->counters + 4, r, nullptr);
    else if (mask)
        k_nvt_two<false, true><<<grid, 256, 0, cs>>>(v4, f4, N, dt, b, h->partials, h->scalars, h->counters + 4, r, mask);
    else
        k_nvt_two<false, false><<<grid, 256, 0, cs>>>(v4, f4, N, dt, b, h->partials, h->scalars, h->counters + 4, r, nullptr);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

extern "C" int cavb200_nvt_step_one(cavb200_handle* h, double* pos, double* vel, const double* force, uint32_t N, double dt,
                                    uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    return nvt_one(h, pos, vel, force, N, dt, group_first, n_group, bussi, nullptr, stream);
    }

extern "C" int cavb200_nvt_step_one_wrap(cavb200_handle* h, double* pos, double* vel, const double* force, int32_t* image,
                                         uint32_t N, double dt, double Lx, double Ly, double Lz, uint32_t group_first,
                                         uint32_t n_group, const cavb200_bussi_args* bussi, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    WrapIn w;
    if (const int rc = make_wrap(w, image, Lx, Ly, Lz))
        return rc;
    return nvt_one(h, pos, vel, force, N, dt, group_first, n_group, bussi, nullptr, stream, &w);
    }

extern "C" int cavb200_nvt_step_two(cavb200_handle* h, double* vel, const double* force, uint32_t N, double dt,
                                    uint32_t group_first, uint32_t n_group, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    return nvt_two(h, vel, force, N, dt, group_first, n_group, nullptr, stream);
    }

extern "C" int cavb200_nvt_step_one_rank1(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                          const double* charge, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                                          uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                                          void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    Rank1In r;
    const int rc = fill_rank1(h, r, charge, pos, L_typeid, couplstr);
    if (rc)
        return rc;
    return nvt_one(h, pos, vel, force_other, N, dt, group_first, n_group, bussi, &r, stream);
    }

extern "C" int cavb200_nvt_step_one_rank1_wrap(cavb200_handle* h, double* pos, double* vel, const double* force_other,
                                               const double* charge, int32_t* image, uint32_t N, double dt, double Lx,
                                               double Ly, double Lz, uint32_t L_typeid, double couplstr,
                                               uint32_t group_first, uint32_t n_group, const cavb200_bussi_args* bussi,
                                               void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    Rank1In r;
    if (const int rc = fill_rank1(h, r, charge, pos, L_typeid, couplstr))
        return rc;
    WrapIn w;
    if (const int rc = make_wrap(w, image, Lx, Ly, Lz))
        return rc;
    return nvt_one(h, pos, vel, force_other, N, dt, group_first, n_group, bussi, &r, stream, &w);
    }

extern "C" int cavb200_nvt_step_two_rank1(cavb200_handle* h, double* vel, const double* force_other, const double* charge,
                                          const double* pos, uint32_t N, double dt, uint32_t L_typeid, double couplstr,
                                          uint32_t group_first, uint32_t n_group, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (N == 0)
        return 0;
    Rank1In r;
    const int rc = fill_rank1(h, r, charge, pos, L_typeid, couplstr);
    if (rc)
        return rc;
    return nvt_two(h, vel, force_other, N, dt, group_first, n_group, &r, stream);
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
    const uint32_t* mask;
    if (!pos || !vel || !charge || !image || !params || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (mis32(pos) || mis32(vel) || mis32(force_other) || (reinterpret_cast<uintptr_t>(image) & 3))
        return (int)cudaErrorMisalignedAddress;
    Rank1In r;
    const int rc = fill_rank1(h, r, charge, pos, L_typeid, params->couplstr);
    if (rc)
        return rc;
    ForceIn fnew = {};
    fnew.pos = reinterpret_cast<const double4*>(pos);
    fnew.charge = charge;
    fnew.image = image;
    fnew.N = N;
    fnew.Lx = Lx;
    fnew.Ly = Ly;
    fnew.Lz = Lz;
    fnew.L_typeid = L_typeid;
    fnew.g = params->couplstr;
    fnew.K = params->K;
    fill_force_constants(fnew);
    BussiIn b = {};
    b.first = group_first;
    b.n = n_group;
    b.rescale = bussi != nullptr && bussi->deltaT != 0.0;
    if (bussi)
        fill_bussi_constants(b, bussi);
    unsigned long long want = ((unsigned long long)N + 255) / 256;
    unsigned long long cap = (unsigned long long)h->num_sms * 3; // one wave of 3 CTAs per SM (85-register budget)
    if (cap > (unsigned long long)MAX_PARTIALS)
        cap = MAX_PARTIALS;
    const int grid = (int)(want < cap ? want : cap);
    WrapIn w = WrapIn();
    if (wrap)
        if (const int rcw = make_wrap(w, const_cast<int32_t*>(image), Lx, Ly, Lz))
            return rcw;
    cudaStream_t cs = (cudaStream_t)stream;
    double4* p4 = (double4*)pos;
    double4* v4 = (double4*)vel;
    const double4* fo4 = (const double4*)force_other;
    Final* fin_out = const_cast<Final*>(rank1_final(h));
    if (wrap && mask)
        k_md_one<true, true><<<grid, 256, 0, cs>>>(p4, v4, fo4, N, dt, b, h->scalars, r, fnew, h->partials, h->counters + 4,
                                                   fin_out, w, mask);
    else if (wrap)
        k_md_one<true, false><<<grid, 256, 0, cs>>>(p4, v4, fo4, N, dt, b, h->scalars, r, fnew, h->partials, h->counters + 4,
                                                    fin_out, w, nullptr);
    else if (mask)
        k_md_one<false, true><<<grid, 256, 0, cs>>>(p4, v4, fo4, N, dt, b, h->scalars, r, fnew, h->partials, h->counters + 4,
                                                    fin_out, w, mask);
    else
        k_md_one<false, false><<<grid, 256, 0, cs>>>(p4, v4, fo4, N, dt, b, h->scalars, r, fnew, h->partials,
                                                     h->counters + 4, fin_out, w, nullptr);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
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
    const uint32_t* mask;
    if (!pos || !vel || !charge || !image || !params || !group_ok(h, N, group_first, n_group, &mask))
        return (int)cudaErrorInvalidValue;
    if (mis32(pos) || mis32(vel) || mis32(force_other) || (reinterpret_cast<uintptr_t>(image) & 3))
        return (int)cudaErrorMisalignedAddress;
    if (!h->coop_supported)
        return (int)cudaErrorNotSupported;
    if (const int fault = check_fault(h))
        return fault;
    Rank1In r;
    int rc = fill_rank1(h, r, charge, pos, L_typeid, params->couplstr);
    if (rc)
        return rc;
    ForceIn fnew = {};
    fnew.pos = reinterpret_cast<const double4*>(pos);
    fnew.charge = charge;
    fnew.image = image;
    fnew.N = N;
    fnew.Lx = Lx;
    fnew.Ly = Ly;
    fnew.Lz = Lz;
    fnew.L_typeid = L_typeid;
    fnew.g = params->couplstr;
    fnew.K = params->K;
    fill_force_constants(fnew);
    BussiIn b = {};
    b.first = group_first;
    b.n = n_group;
    b.rescale = bussi != nullptr && bussi->deltaT != 0.0;
    if (bussi)
        fill_bussi_constants(b, bussi);
    const void* kern;
    int threads, per_sm_want;
    WrapIn w = WrapIn();
    if (wrap)
        if (const int rcw = make_wrap(w, const_cast<int32_t*>(image), Lx, Ly, Lz))
            return rcw;
    switch (h->tune.md_shape)
        {
    case 1:
        if (mask)
            kern = wrap ? (const void*)k_md_fused<384, 1, true, true> : (const void*)k_md_fused<384, 1, false, true>;
        else
            kern = wrap ? (const void*)k_md_fused<384, 1, true, false> : (const void*)k_md_fused<384, 1, false, false>;
        threads = 384;
        per_sm_want = 2;
        break;
    default: // folder CTA alone on its SM
        if (mask)
            kern = wrap ? (const void*)k_md_fused<768, 1, true, true> : (const void*)k_md_fused<768, 1, false, true>;
        else
            kern = wrap ? (const void*)k_md_fused<768, 1, true, false> : (const void*)k_md_fused<768, 1, false, false>;
        threads = 768;
        per_sm_want = 1;
        break;
        }
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
    void* args[] = {&p4, &v4, &fo4, &N, &dt, &b, &r, &fnew, &recsF, &recsB, &finals, &sca, &ctr, &fin_out, &w, &mask};
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
    if (mis32(net_force))
        return (int)cudaErrorMisalignedAddress;
    Rank1In r;
    const int rc = fill_rank1(h, r, charge, pos, L_typeid, couplstr);
    if (rc)
        return rc;
    unsigned long long want = ((unsigned long long)N + 255) / 256;
    const unsigned long long cap = (unsigned long long)h->num_sms * 8;
    k_net_force_add_rank1<<<(int)(want < cap ? want : cap), 256, 0, (cudaStream_t)stream>>>((double4*)net_force, N, r);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
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
        const unsigned long long want = ((unsigned long long)n + 255) / 256;
        const unsigned long long cap = (unsigned long long)h->num_sms * 8;
        k_group_mask<<<(int)(want < cap ? want : cap), 256, 0, cs>>>(group_idx, n, N, h->group_mask, bad);
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
    if (mis32(pos))
        return (int)cudaErrorMisalignedAddress;
    if (N == 0)
        return 0;
    cudaStream_t cs = (cudaStream_t)stream;
    unsigned long long* sc = h->counters + 49; // {first, count, ticket}
    CAVB_CHECK(cudaMemsetAsync(sc, 0xFF, sizeof(unsigned long long), cs));
    CAVB_CHECK(cudaMemsetAsync(sc + 1, 0, 2 * sizeof(unsigned long long), cs));
    const unsigned long long want = ((unsigned long long)N + 255) / 256;
    const unsigned long long cap = (unsigned long long)h->num_sms * 8;
    k_photon_reindex<<<(int)(want < cap ? want : cap), 256, 0, cs>>>(reinterpret_cast<const double4*>(pos), N, L_typeid, sc,
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
