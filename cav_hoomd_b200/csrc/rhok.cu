// rhok.cu -- F(k,t): the density field rho[t][k] = sum_j exp(i k.r_j(t)) for a batch of frames,
// and the origin/lag correlation F = mean_k Re(rho_0 conj(rho_t)).
//
// Batched form of compute_density_field / compute_field_autocorr
// (reference src/cavitymd/analysis.py:34-47, :359-364), which loops over k in Python and makes K
// NumPy passes over N every step.  Here one launch covers T frames x K wavevectors:
//   grid (P, T): CTA (p, t) owns a contiguous slice of frame t's particles; tiles of positions are
//   copied into shared memory one tile ahead (cp.async, two buffers); thread (group, k-quad) keeps
//   four rho_k's (re, im) in registers and walks the tile's particles group, group+G, ... (broadcast
//   LDS); groups are folded in shared memory; slices are folded by a second tiny kernel in slice order.
// The sum order is fixed, so results are bitwise reproducible.  The work is FP64 bound (17 fp64
// instructions per (particle, k) pair against 24/K bytes), not HBM bound, and the contraction is
// only k x 3 deep: no tensor-core shape here (BASELINE.json north_star (3)).
#include "cavb200_internal.cuh"

namespace cavb
    {
#ifndef RHOK_MIN_CTAS
#define RHOK_MIN_CTAS 2
#endif

#ifndef RHOK_KB
#define RHOK_KB 4
#endif
#ifndef RHOK_GRID_PER_SM
#define RHOK_GRID_PER_SM 24 // most CTAs of a launch per resident slot (rhok_slices picks the count)
#endif
#ifndef RHOK_CTA
#define RHOK_CTA 256 // largest (and default) CTA size
#endif
constexpr int RHOK_KB_HOST = RHOK_KB;
#ifndef RHOK_TILE_N
#define RHOK_TILE_N 512
#endif
constexpr int RHOK_TILE = RHOK_TILE_N;  // particles per shared-memory tile (16 KB as double4; two buffers)
constexpr uint32_t RHOK_F32 = 13;  // internal `stride` code: float32 xyz positions (frame_stride then counts floats)

// exp(i x) for |x| < 2^20 by table and short polynomial, both components to ~1 ulp of 1 (abs. error <= 2.4e-16).
// History (DESIGN.md 3.4): the library sincos() cost ~70 issue slots per call and left the kernel issue bound; an inline
// quadrant reduction with fdlibm's degree-13/14 polynomials brought a (particle, k) pair to 27 FP64 instructions and the
// FP64 pipe to 79 % busy -- from there the only way down is fewer FP64 instructions.  Now:
//   n = rint(x * 512/2pi) by the 1.5*2^52 trick;  r = x - n*(2pi/512) with a two-FMA Cody-Waite reduction, |r| <= pi/512;
//   (C, S) = (cos, sin)(2pi (n mod 512)/512) from a 512-entry table (host long double, rounded once, built by octant
//   symmetry so the axes are exact);  sin r = r - r^3/6 + r^5/120 (truncation 1e-17 relative),  cos r = 1 - z/2 + c4 z^2
//   with c4 shifted off 1/24 so the dropped z^3/720 is spread over [0, (pi/512)^2] (2e-17 absolute);  and the rotation
//   re += c C - s S,  im += c S + s C  is the accumulate itself: 17 FP64 instructions per pair instead of 27, and the ten
//   integer / select instructions of a quadrant fix-up are one mask and one address.
// The table sits in shared memory EIGHT times, interleaved by 16 bytes: lane l reads copy l & 7, so the eight lanes of a
// quarter warp -- the unit a 128-bit shared load is served in -- hit eight different bank groups whatever their entries
// are: one conflict-free LDS.128 per pair (four wavefronts) where a single copy would serialise ~2.5-fold and make the
// shared-memory pipe, not the FP64 pipe, the limit.
// (the constants sit in constant memory so that every DFMA takes its coefficient as a c[bank][offset] operand)
constexpr int RHOK_TAB = 512;  // table entries over one turn
constexpr int RHOK_REP = 8;    // interleaved copies
__constant__ double SC[9] = {
    6755399441055744.0,                       // 0  1.5 * 2^52
    6.36619772367581382433e-01 * 128.0,       // 1  512 / 2pi   (fl(2/pi) * 2^7, exact scaling)
    1.57079632679489655800e+00 / 128.0,       // 2  2pi/512 hi  (fl(pi/2) * 2^-7)
    6.12323399573676603587e-17 / 128.0,       // 3  2pi/512 lo
    8.33333333333333333333e-03,               // 4  1/120
    -1.66666666666666666667e-01,              // 5  -1/6
    4.16666666666666666667e-02 - 0.8 * 3.764955292163604e-05 / 720.0, // 6  1/24 - 0.8 (pi/512)^2 / 720
    -0.5, 1.0};
// sin and cos of the REDUCED argument r = x - n 2pi/512 and the turn count n (two's complement, only n & 511 matters)
__device__ __forceinline__ void sincos_reduced(double x, double& sr, double& cr, int& n)
    {
    const double t = __fma_rn(x, SC[1], SC[0]);
    n = __double2loint(t);
    const double nf = __dadd_rn(t, -SC[0]);
    double r = __fma_rn(-nf, SC[2], x);
    r = __fma_rn(-nf, SC[3], r);
    const double z = __dmul_rn(r, r);
    sr = __fma_rn(__dmul_rn(r, z), __fma_rn(z, SC[4], SC[5]), r);
    cr = __fma_rn(z, __fma_rn(z, SC[6], SC[7]), SC[8]);
    }

__device__ __forceinline__ unsigned int abs_hi(double v) { return (unsigned int)__double2hiint(v) & 0x7fffffffu; }

// One thread's walk over a staged tile: particles pg, pg + groups, ... against its KB wave vectors.
// CHECK = false: the caller has bounded every |k.r| of the tile below 2^20, so the inner loop carries no range test
// (2-3 integer instructions per (particle, k) pair that share the issue port with the half-rate FP64 pipe).
// `tab` is the interleaved table, entry e of copy c at byte (e * RHOK_REP + c) * 16; lane_slot = (lane & 7) * 16.
template<int KB, bool CHECK>
__device__ __forceinline__ void rhok_walk(const double4* tile, const char* tab, uint32_t lane_slot, uint32_t pg,
                                          uint32_t n, uint32_t groups, const double (&kx)[KB], const double (&ky)[KB],
                                          const double (&kz)[KB], double (&re)[KB], double (&im)[KB])
    {
    for (uint32_t j = pg; j < n; j += groups)
        {
        const double4 rj = tile[j]; // one broadcast LDS.128 (a warp holds two neighbouring particle groups)
        const double x = rj.x, y = rj.y, z = rj.z;
        double kr[KB];
        bool huge = false;
#pragma unroll
        for (int m = 0; m < KB; m++)
            {
            // analysis.py:42 np.dot(positions, k_vec) = x kx + y ky + z kz (NumPy hands this to a BLAS
            // gemv, which contracts to FMAs on any AVX2 host; so does this)
            kr[m] = __fma_rn(z, kz[m], __fma_rn(y, ky[m], __dmul_rn(x, kx[m])));
            // |kr| >= 2^20, inf or nan: exponent test on the integer pipe (DSETP would sit on the FP64 pipe)
            if (CHECK)
                huge = huge || (__double2hiint(kr[m]) & 0x7fffffff) >= 0x41300000;
            }
        if (!CHECK || !huge)
            {
            // one basic block for the KB independent chains: coefficients are fetched once
            // (tried and dropped: the chains written stage by stage -- spills; the next particle's arguments formed
            // beside the chains of this one, a software pipeline -- 124 registers, 0.0816 ms per frame against 0.0810; only
            // the next particle's coordinates loaded an iteration ahead -- 0.0828 against 0.0794)
#pragma unroll
            for (int m = 0; m < KB; m++)
                {
                double sr, cr;
                int q;
                sincos_reduced(kr[m], sr, cr, q);
                // byte offset of entry q mod 512, copy lane & 7: one shift, one (and, or), the table base rides in the LDS itself
                const double2 w = *reinterpret_cast<const double2*>(
                    tab + ((((uint32_t)q << 7) & ((RHOK_TAB - 1u) << 7)) | lane_slot));
                re[m] = __fma_rn(-sr, w.y, __fma_rn(cr, w.x, re[m]));
                im[m] = __fma_rn(cr, w.y, __fma_rn(sr, w.x, im[m]));
                }
            }
        else
            {
            for (int m = 0; m < KB; m++)
                {
                double sn, cs;
                sincos(kr[m], &sn, &cs); // huge arguments (and inf/nan): the library's Payne-Hanek path
                re[m] += cs;
                im[m] += sn;
                }
            }
        }
    }

// asynchronous global -> shared copies (LDGSTS): the tile of the NEXT iteration lands while this one is walked
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
    {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned int)__cvta_generic_to_shared(smem)), "l"(gmem)
                 : "memory");
    }
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem)
    {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned int)__cvta_generic_to_shared(smem)), "l"(gmem)
                 : "memory");
    }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Stage tile `tile` of a frame into `dst` as double4 {x, y, z, -}.  Double positions (Scalar4 or xyz) are copied
// asynchronously, 16 or 8 bytes at a time, with no register in between; float32 positions are widened on the way
// (exactly, as NumPy does in np.dot(f32, f64)) and therefore go through registers, synchronously.
__device__ __forceinline__ void rhok_stage(double4* dst, const double* pos, uint32_t stride, unsigned long long frame_off,
                                           uint32_t base, uint32_t n, uint32_t tid, uint32_t nthreads)
    {
    if (stride == 4)
        {
        const double2* src = reinterpret_cast<const double2*>(pos + frame_off) + 2ull * base;
        double2* d2 = reinterpret_cast<double2*>(dst);
        for (uint32_t e = tid; e < 2 * n; e += nthreads)
            cp_async16(d2 + e, src + e);
        }
    else if (stride == RHOK_F32)
        {
        const float* src = reinterpret_cast<const float*>(pos) + frame_off + 3ull * base;
        double* d1 = reinterpret_cast<double*>(dst);
        for (uint32_t e = tid; e < 3 * n; e += nthreads)
            {
            const uint32_t j = e / 3, c = e - 3 * j;
            d1[4 * j + c] = (double)__ldg(src + e);
            }
        }
    else
        {
        const double* src = pos + frame_off + 3ull * base;
        double* d1 = reinterpret_cast<double*>(dst);
        for (uint32_t e = tid; e < 3 * n; e += nthreads)
            {
            const uint32_t j = e / 3, c = e - 3 * j;
            cp_async8(d1 + 4 * j + c, src + e);
            }
        }
    cp_async_commit();
    }

// grid (P, T); thread (pg, kq): particle group pg walks the tile with stride `groups`, kq owns KB
// consecutive wave vectors whose components and (re, im) accumulators live in registers, so the one
// shared-memory load and the loop bookkeeping of a particle are paid once per KB (particle, k) pairs.
// Two tile buffers: the copy of tile i+1 is issued before tile i is walked, so no warp ever waits for HBM -- with two
// CTAs of eight warps per SM, a CTA that stopped to stage its next tile left the FP64 pipe to the other CTA's two warps
// per scheduler, which cannot keep it busy.
// F32: the instantiation for float32 positions (its six prefetch registers cost the double instantiation 3.7 % when
// both lived in one kernel: 0.0809 -> 0.0839 ms per frame).
template<int KB, bool F32>
__global__ void __launch_bounds__(RHOK_CTA, RHOK_MIN_CTAS)
    k_rhok(const double* __restrict__ pos, uint32_t stride, unsigned long long frame_stride, uint32_t N,
           const double* __restrict__ kvec, uint32_t k0, uint32_t Ks, uint32_t K, double* __restrict__ out, uint32_t P,
           int direct, const double2* __restrict__ table)
    {
    __shared__ unsigned int tile_maxhi[2]; // largest hi word of |coordinate| in a staged tile (by buffer)
    extern __shared__ double2 stab[];      // [RHOK_TAB][RHOK_REP] (cos, sin)(2 pi e / RHOK_TAB), then the two tile buffers
    double4* tiles2 = reinterpret_cast<double4*>(stab + RHOK_TAB * RHOK_REP); // [2][RHOK_TILE]
    double* sred = reinterpret_cast<double*>(tiles2); // [groups][KQ * KB][2], after the last tile has been walked

    const uint32_t t = blockIdx.y, p = blockIdx.x;
    const uint32_t tid = threadIdx.x;
    const uint32_t KQ = (Ks + KB - 1) / KB;      // k-quads of this slab (host guarantees KQ <= blockDim.x)
    const uint32_t groups = blockDim.x / KQ;
    const uint32_t kq = tid % KQ, pg = tid / KQ;
    const bool active = pg < groups;

    // contiguous slice of this frame, in whole tiles
    const uint32_t tiles = (N + RHOK_TILE - 1) / RHOK_TILE;
    const uint32_t tiles_per = (tiles + P - 1) / P;
    const uint32_t tile_lo = p * tiles_per;
    const uint32_t tile_hi = min(tiles, tile_lo + tiles_per);
    const unsigned long long frame_off = (unsigned long long)t * frame_stride;

    // every copy of a table entry is written by one thread: consecutive threads write consecutive 16-byte slots.
    // Programmatic dependent launch: the table (handle-owned, constant) may be read while the previous kernel of the
    // stream is still draining; positions, wave vectors and the partial sums may not be touched before pdl_wait()
    for (uint32_t e = tid; e < RHOK_TAB * RHOK_REP; e += blockDim.x)
        stab[e] = __ldg(table + e / RHOK_REP);
    pdl_wait();
    if (tile_lo < tile_hi)
        rhok_stage(tiles2, pos, stride, frame_off, tile_lo * RHOK_TILE, min((uint32_t)RHOK_TILE, N - tile_lo * RHOK_TILE), tid,
                   blockDim.x);

    double kx[KB], ky[KB], kz[KB], re[KB], im[KB];
#pragma unroll
    for (int m = 0; m < KB; m++)
        {
        const uint32_t k = kq * KB + m;
        const bool in = active && k < Ks;
        kx[m] = in ? __ldg(kvec + 3 * (k0 + k) + 0) : 0.0;
        ky[m] = in ? __ldg(kvec + 3 * (k0 + k) + 1) : 0.0;
        kz[m] = in ? __ldg(kvec + 3 * (k0 + k) + 2) : 0.0;
        re[m] = im[m] = 0.0;
        }
    double kbound = 0.0; // max over this thread's wave vectors of |kx| + |ky| + |kz| >= |k.r| / max|coordinate|
#pragma unroll
    for (int m = 0; m < KB; m++)
        kbound = fmax(kbound, fabs(kx[m]) + fabs(ky[m]) + fabs(kz[m]));
    if (tid < 2)
        tile_maxhi[tid] = 0u;
    const char* tab = reinterpret_cast<const char*>(stab);
    const uint32_t lane_slot = (tid & (RHOK_REP - 1)) * 16u;

    constexpr int RHOK_PF = (3 * RHOK_TILE + 255) / 256; // floats of a tile per thread of a 256-thread CTA
    float pf[RHOK_PF]; // (dead in the double instantiation)
    const bool pre32 = F32 && blockDim.x * (uint32_t)RHOK_PF >= 3u * RHOK_TILE;
    for (uint32_t tile = tile_lo; tile < tile_hi; tile++)
        {
        const uint32_t cur = (tile - tile_lo) & 1u;
        const double4* buf = tiles2 + cur * RHOK_TILE;
        const uint32_t n = min((uint32_t)RHOK_TILE, N - tile * RHOK_TILE);
        cp_async_wait_all();
        __syncthreads(); // this tile has landed (and the table, first time); everyone has left the other buffer
        uint32_t n_next = 0u;
        if constexpr (!F32)
            {
            if (tile + 1 < tile_hi)
                rhok_stage(tiles2 + (cur ^ 1u) * RHOK_TILE, pos, stride, frame_off, (tile + 1) * RHOK_TILE,
                           min((uint32_t)RHOK_TILE, N - (tile + 1) * RHOK_TILE), tid, blockDim.x);
            }
        else
            {
            n_next = tile + 1 < tile_hi ? min((uint32_t)RHOK_TILE, N - (tile + 1) * RHOK_TILE) : 0u;
            if (pre32)
                {
                // float32 positions cannot be copied asynchronously (they are widened on the way): this thread's six
                // floats of the next tile wait in registers while this tile is walked
                const float* src = reinterpret_cast<const float*>(pos) + frame_off + 3ull * (tile + 1) * RHOK_TILE;
#pragma unroll
                for (int i = 0; i < RHOK_PF; i++)
                    {
                    const uint32_t e = tid + i * blockDim.x;
                    pf[i] = e < 3 * n_next ? __ldg(src + e) : 0.0f;
                    }
                }
            else if (n_next)
                rhok_stage(tiles2 + (cur ^ 1u) * RHOK_TILE, pos, stride, frame_off, (tile + 1) * RHOK_TILE, n_next, tid,
                           blockDim.x);
            }
        unsigned int mx = 0u; // largest hi word of |coordinate| among the particles this thread looks at
        for (uint32_t j = tid; j < n; j += blockDim.x)
            {
            const double4 r = buf[j];
            mx = max(mx, max(max(abs_hi(r.x), abs_hi(r.y)), abs_hi(r.z)));
            }
        mx = __reduce_max_sync(0xffffffffu, mx);
        if ((tid & 31u) == 0)
            atomicMax(&tile_maxhi[cur], mx);
        __syncthreads();
        // upper bound of |coordinate| over the tile (hi word + 1, lo word 0 bounds every double with that hi word); with
        // the thread's own bound on |kx| + |ky| + |kz| it decides once per tile whether any argument can reach 2^20
        const unsigned int mh = tile_maxhi[cur];
        if (tid == 0)
            tile_maxhi[cur ^ 1u] = 0u;
        const bool fast = mh < 0x7ff00000u && __dmul_rn(kbound, __hiloint2double((int)(mh + 1u), 0)) < 1048575.0;
        if (active)
            {
            if (fast)
                rhok_walk<KB, false>(buf, tab, lane_slot, pg, n, groups, kx, ky, kz, re, im);
            else
                rhok_walk<KB, true>(buf, tab, lane_slot, pg, n, groups, kx, ky, kz, re, im);
            }
        if constexpr (F32)
            {
            if (pre32)
                {
                double* d1 = reinterpret_cast<double*>(tiles2 + (cur ^ 1u) * RHOK_TILE); // nobody reads this buffer now
#pragma unroll
                for (int i = 0; i < RHOK_PF; i++)
                    {
                    const uint32_t e = tid + i * blockDim.x;
                    const uint32_t j = e / 3, c = e - 3 * j;
                    if (e < 3 * n_next)
                        d1[4 * j + c] = (double)pf[i];
                    }
                }
            }
        }
    pdl_launch_dependents(); // the fold kernel's (or the next call's) CTAs may take the SMs this grid's CTAs leave
    __syncthreads(); // the tile buffers become the fold area

    // fold the particle groups (fixed order)
    const uint32_t KP = KQ * KB;
    if (active)
        {
#pragma unroll
        for (int m = 0; m < KB; m++)
            {
            sred[(pg * KP + kq * KB + m) * 2 + 0] = re[m];
            sred[(pg * KP + kq * KB + m) * 2 + 1] = im[m];
            }
        }
    __syncthreads();
    for (uint32_t k = tid; k < Ks; k += blockDim.x)
        {
        double r = 0.0, i = 0.0;
        for (uint32_t g = 0; g < groups; g++)
            {
            r += sred[(g * KP + k) * 2 + 0];
            i += sred[(g * KP + k) * 2 + 1];
            }
        double* dst = direct ? out + ((unsigned long long)t * K + k0 + k) * 2
                             : out + (((unsigned long long)t * P + p) * K + k0 + k) * 2;
        dst[0] = r;
        dst[1] = i;
        }
    }

// one warp per (t, k): lane L adds slices L, L + 32, ... (independent loads), then a fixed shuffle tree
__global__ void k_rhok_fold(const double* __restrict__ part, uint32_t P, uint32_t K, uint32_t T, double* __restrict__ rho)
    {
    const unsigned long long e = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; // (t, k) pair
    const uint32_t lane = threadIdx.x & 31;
    pdl_wait(); // launched while k_rhok was draining
    pdl_launch_dependents();
    if (e >= (unsigned long long)T * K)
        return;
    const unsigned long long t = e / K, k = e % K;
    double r = 0.0, i = 0.0;
    for (uint32_t p = lane; p < P; p += 32)
        {
        const double2 v = *reinterpret_cast<const double2*>(part + ((t * P + p) * K + k) * 2);
        r += v.x;
        i += v.y;
        }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1)
        {
        r += __shfl_xor_sync(0xffffffffu, r, m);
        i += __shfl_xor_sync(0xffffffffu, i, m);
        }
    if (lane == 0)
        {
        rho[e * 2 + 0] = r;
        rho[e * 2 + 1] = i;
        }
    }

// mean_k Re(a_k conj(b_k)) of two fields of K {re, im} pairs, k ascending (analysis.py:361:
// np.mean(np.real(f0 * np.conj(ft)))).  The one loop of k_fkt and k_fkt_track, so that both give the same bits.
__device__ __forceinline__ double fkt_pair(const double* a, const double* b, uint32_t K)
    {
    double acc = 0.0;
    for (uint32_t k = 0; k < K; k++)
        {
        // Re((ar + i ai)(br - i bi)) = ar br + ai bi
        acc += a[2 * k] * b[2 * k] + a[2 * k + 1] * b[2 * k + 1];
        }
    return acc / (double)K;
    }

// F[o][l] = mean_k Re(rho[o][k] conj(rho[o+l][k]))
__global__ void k_fkt(const double* __restrict__ rho, uint32_t T, uint32_t K, uint32_t n_origins, uint32_t n_lags,
                      double* __restrict__ out)
    {
    const unsigned long long e = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (unsigned long long)n_origins * n_lags)
        return;
    const unsigned long long o = e / n_lags, l = e % n_lags;
    if (o + l >= T)
        {
        out[e] = __longlong_as_double(0x7ff8000000000000ll);
        return;
        }
    out[e] = fkt_pair(rho + o * K * 2, rho + (o + l) * K * 2, K);
    }

// F(k,t) tracker step (cavb200_fkt_track_step): after k_rhok (and k_rhok_fold) have written this frame's rho into the
// slot, one CTA appends the record {timestep, n_refs, F of every stored reference against rho (NaN past n_refs), rho}
// to the ring (RECORD) and/or copies rho into reference slot n_refs (ADD_REFERENCE).  Thread j < max_refs forms F of
// reference j with the loop k_fkt uses, so a record is bit-identical to cavb200_fkt on (reference j, this frame).
__global__ void k_fkt_track(const double* __restrict__ rho, double* __restrict__ refs, uint32_t K, uint32_t max_refs,
                            uint32_t n_refs, uint32_t flags, double timestep, double* __restrict__ ring,
                            unsigned long long* __restrict__ count, unsigned long long capacity)
    {
    const uint32_t tid = threadIdx.x;
    pdl_wait(); // rho is written by the launch before this one
    pdl_launch_dependents();
    if (flags & CAVB200_FKT_RECORD)
        {
        const unsigned long long n = *count;
        double* r = ring + (n % capacity) * (2ull + max_refs + 2ull * K);
        if (tid == 0)
            {
            r[0] = timestep;
            r[1] = (double)n_refs;
            }
        for (uint32_t j = tid; j < max_refs; j += blockDim.x)
            r[2 + j] = j < n_refs ? fkt_pair(refs + 2ull * K * j, rho, K) : __longlong_as_double(0x7ff8000000000000ll);
        for (uint32_t e = tid; e < 2 * K; e += blockDim.x)
            r[2 + max_refs + e] = rho[e];
        __syncthreads(); // every thread has read the counter
        if (tid == 0)
            *count = n + 1;
        }
    if (flags & CAVB200_FKT_ADD_REFERENCE)
        for (uint32_t e = tid; e < 2 * K; e += blockDim.x)
            refs[2ull * K * n_refs + e] = rho[e];
    }
    } // namespace cavb

using namespace cavb;

// (cos, sin)(2 pi e / RHOK_TAB) in long double, rounded once; octant symmetry makes cos^2 + sin^2 symmetric over the turn
// and the four axis entries exactly (+-1, 0), (0, +-1)
static void rhok_table_host(double2* tab)
    {
    const long double two_pi = 6.283185307179586476925286766559005768L;
    const int Q = RHOK_TAB / 4;
    for (int e = 0; e < RHOK_TAB; e++)
        {
        const int quad = e / Q, j = e % Q;
        long double c, s;
        if (j <= Q / 2)
            {
            c = cosl(two_pi * j / RHOK_TAB);
            s = sinl(two_pi * j / RHOK_TAB);
            }
        else
            {
            c = sinl(two_pi * (Q - j) / RHOK_TAB);
            s = cosl(two_pi * (Q - j) / RHOK_TAB);
            }
        const double cd = (double)c, sd = (double)s;
        tab[e] = quad == 0 ? make_double2(cd, sd)
                           : (quad == 1 ? make_double2(-sd, cd) : (quad == 2 ? make_double2(-cd, -sd) : make_double2(sd, -cd)));
        }
    }

// How many slices P a frame is cut into.  The CTAs of a launch do equal work and two are resident per SM, so they run
// in waves: the launch takes ceil(P T / slots) waves of ceil(tiles / P) tiles each, plus a fixed cost per CTA (table
// fill, fold: about a quarter of a tile).  A fixed 24 CTAs per SM lost 2-4 % to a ragged last wave or a ragged last
// tile count (1M particles: 32 frames P = 111 -> 12 waves x 18 tiles = 216 tile times against 211.2 ideal, P = 37 -> 4 x
// 53 = 212; 8 frames: P = 444 -> 12 x 5 = 60 against 52.8, P = 222 -> 6 x 9 = 54; profiles/fkt_r2c.txt).
static uint32_t rhok_slices(uint32_t tiles, uint32_t T, uint32_t slots)
    {
    uint32_t pmax = (uint32_t)(((uint64_t)RHOK_GRID_PER_SM * slots + T - 1) / T);
    if (pmax > tiles)
        pmax = tiles;
    if (pmax < 1)
        pmax = 1;
    uint32_t best = 1;
    double best_cost = 0.0;
    for (uint32_t P = 1; P <= pmax; P++)
        {
        const uint64_t waves = ((uint64_t)P * T + slots - 1) / slots;
        const uint32_t per = (tiles + P - 1) / P;
        const double cost = (double)waves * ((double)per + 0.25);
        if (P == 1 || cost < best_cost)
            {
            best = P;
            best_cost = cost;
            }
        }
    return best;
    }

// First use on a handle: the 8 KB table (a blocking copy from pageable memory, like the workspace growth in rhok_launch)
// and the kernels' shared-memory limit.
static int rhok_table_init(cavb200_handle* h)
    {
    if (h->rhok_table)
        return 0;
    double2 host_tab[RHOK_TAB];
    rhok_table_host(host_tab);
    CAVB_CHECK(cudaMalloc((void**)&h->rhok_table, sizeof(host_tab)));
    CAVB_CHECK(cudaMemcpy(h->rhok_table, host_tab, sizeof(host_tab), cudaMemcpyHostToDevice));
    const int smem_max = (int)(sizeof(double2) * RHOK_TAB * RHOK_REP + sizeof(double4) * 2 * RHOK_TILE);
    CAVB_CHECK(cudaFuncSetAttribute(k_rhok<RHOK_KB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    CAVB_CHECK(cudaFuncSetAttribute(k_rhok<RHOK_KB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    return 0;
    }

// Everything rhok_launch would set up on first use for one frame (T = 1) of at most N particles and K wave vectors:
// the table and a slice workspace no such call outgrows.  rhok_slices is not monotonic in the tile count, so the
// workspace is sized for its upper limit min(tiles, RHOK_GRID_PER_SM * slots), which covers every N' <= N.  Blocking.
static int rhok_prime(cavb200_handle* h, uint32_t N, uint32_t K)
    {
    if (const int err = rhok_table_init(h))
        return err;
    const uint64_t tiles = ((uint64_t)N + RHOK_TILE - 1) / RHOK_TILE;
    const uint64_t pmax = (uint64_t)RHOK_GRID_PER_SM * 2u * (uint64_t)h->num_sms;
    const uint64_t P = tiles < pmax ? tiles : pmax;
    const uint64_t need = P > 1 ? sizeof(double) * 2ull * K * P : 0;
    if (h->rhok_partials_bytes < need)
        {
        CAVB_CHECK(cudaDeviceSynchronize());
        cudaFree(h->rhok_partials);
        h->rhok_partials = nullptr;
        h->rhok_partials_bytes = 0;
        CAVB_CHECK(cudaMalloc((void**)&h->rhok_partials, need));
        h->rhok_partials_bytes = need;
        }
    return 0;
    }

static int rhok_launch(cavb200_handle* h, const double* pos, uint32_t stride, uint64_t frame_stride, uint32_t N,
                       uint32_t T, const double* kvec, uint32_t K, double* rho, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (T == 0 || K == 0)
        return 0;
    if (!kvec || !rho || (N > 0 && !pos) || (stride != 3 && stride != 4 && stride != RHOK_F32))
        return (int)cudaErrorInvalidValue;
    if (stride == 4 && ((reinterpret_cast<uintptr_t>(pos) & 31) || (frame_stride & 3)))
        return (int)cudaErrorMisalignedAddress;
    if (stride == RHOK_F32 && (reinterpret_cast<uintptr_t>(pos) & 3))
        return (int)cudaErrorMisalignedAddress;
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0)
        {
        CAVB_CHECK(cudaMemsetAsync(rho, 0, sizeof(double) * 2ull * K * T, s));
        return 0;
        }
    if (const int err = rhok_table_init(h))
        return err;
    // two CTAs of 256 threads per SM: the 64 KB table of each leaves no room for four of 128 (which were worth 1-2 % when
    // the table was four entries: a CTA staging its next tile idled a quarter of the SM's warps instead of half)
    const int threads = (h->tune.rhok_threads >= 128 && h->tune.rhok_threads <= RHOK_CTA && h->tune.rhok_threads % 128 == 0)
                            ? h->tune.rhok_threads
                            : RHOK_CTA;
    const uint32_t tiles = (N + RHOK_TILE - 1) / RHOK_TILE;
    const uint32_t slots = 2u * (uint32_t)h->num_sms;
    // grid y is at most 65535: frames go in chunks of that many, each with its own slice count.  Chunks after the first
    // start at offset pointers (frame_stride doubles -- floats on the float32 path, whose pointer travels as a double*
    // -- per frame, 2K doubles of rho per frame), so the kernels never see more than one chunk.  Consecutive chunks reuse
    // the workspace in stream order: k_rhok touches it only after pdl_wait(), i.e. after the previous fold has finished.
    constexpr uint32_t TCHUNK = 65535;
    uint64_t need = 0;
    for (uint32_t t0 = 0; t0 < T; t0 += TCHUNK)
        {
        const uint32_t Tc = (T - t0) < TCHUNK ? (T - t0) : TCHUNK;
        const uint32_t P = rhok_slices(tiles, Tc, slots);
        if (P > 1 && sizeof(double) * 2ull * K * Tc * P > need)
            need = sizeof(double) * 2ull * K * Tc * P;
        }
    if (h->rhok_partials_bytes < need)
        {
        // growing the workspace is the one place a call may synchronise (first call / larger batch)
        CAVB_CHECK(cudaStreamSynchronize(s));
        cudaFree(h->rhok_partials);
        h->rhok_partials = nullptr;
        h->rhok_partials_bytes = 0;
        CAVB_CHECK(cudaMalloc((void**)&h->rhok_partials, need));
        h->rhok_partials_bytes = need;
        }
    cudaLaunchAttribute pdl_attr;
    pdl_attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl_attr.val.programmaticStreamSerializationAllowed = 1;
    // wave vectors in slabs of at most threads*KB = 1024 (one launch for the usual K); KB = 4 k per thread
#ifndef RHOK_KB
#define RHOK_KB 4
#endif
    constexpr int KB = RHOK_KB;
    for (uint32_t t0 = 0; t0 < T; t0 += TCHUNK)
        {
        const uint32_t Tc = (T - t0) < TCHUNK ? (T - t0) : TCHUNK;
        const uint32_t P = rhok_slices(tiles, Tc, slots);
        const int direct = (P == 1);
        const double* pos_c = stride == RHOK_F32
                                  ? reinterpret_cast<const double*>(reinterpret_cast<const float*>(pos) + t0 * frame_stride)
                                  : pos + t0 * frame_stride;
        double* rho_c = rho + 2ull * K * t0;
        double* target = direct ? rho_c : h->rhok_partials;
        for (uint32_t k0 = 0; k0 < K; k0 += (uint32_t)threads * KB)
            {
            const uint32_t Ks = (K - k0) < (uint32_t)threads * KB ? (K - k0) : (uint32_t)threads * KB;
            // table | two tile buffers (32 KB; the fold of the particle groups reuses them: 2 * groups * KQ * KB doubles <= 16 KB)
            const size_t smem = sizeof(double2) * RHOK_TAB * RHOK_REP + sizeof(double4) * 2 * RHOK_TILE;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(P, Tc);
            cfg.blockDim = dim3(threads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = s;
            cfg.attrs = &pdl_attr;
            cfg.numAttrs = h->tune.pdl ? 1 : 0;
            unsigned long long fs = frame_stride;
            const double2* tabp = (const double2*)h->rhok_table;
            int direct_i = direct;
            void* args[] = {(void*)&pos_c, (void*)&stride, (void*)&fs,     (void*)&N, (void*)&kvec,     (void*)&k0,
                            (void*)&Ks,    (void*)&K,      (void*)&target, (void*)&P, (void*)&direct_i, (void*)&tabp};
            CAVB_CHECK(cudaLaunchKernelExC(&cfg, stride == RHOK_F32 ? (const void*)k_rhok<KB, true> : (const void*)k_rhok<KB, false>,
                                           args));
            h->launches += 1;
            }
        if (!direct)
            {
            const unsigned long long pairs = (unsigned long long)Tc * K;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned int)((pairs * 32 + 255) / 256));
            cfg.blockDim = dim3(256);
            cfg.stream = s;
            cfg.attrs = &pdl_attr;
            cfg.numAttrs = h->tune.pdl ? 1 : 0;
            const double* part = target;
            void* args[] = {(void*)&part, (void*)&P, (void*)&K, (void*)&Tc, (void*)&rho_c};
            CAVB_CHECK(cudaLaunchKernelExC(&cfg, (const void*)k_rhok_fold, args));
            h->launches += 1;
            }
        }
    return 0;
    }

extern "C" int cavb200_rhok(cavb200_handle* h, const double* pos, uint32_t stride, uint64_t frame_stride, uint32_t N,
                            uint32_t T, const double* kvec, uint32_t K, double* rho, void* stream)
    {
    if (stride != 3 && stride != 4)
        return (int)cudaErrorInvalidValue;
    return rhok_launch(h, pos, stride, frame_stride, N, T, kvec, K, rho, stream);
    }

extern "C" int cavb200_rhok_f32(cavb200_handle* h, const float* pos_xyz, uint64_t frame_stride, uint32_t N, uint32_t T,
                                const double* kvec, uint32_t K, double* rho, void* stream)
    {
    return rhok_launch(h, reinterpret_cast<const double*>(pos_xyz), RHOK_F32, frame_stride, N, T, kvec, K, rho, stream);
    }

extern "C" int cavb200_fkt(cavb200_handle* h, const double* rho, uint32_t T, uint32_t K, uint32_t n_origins,
                           uint32_t n_lags, double* out, void* stream)
    {
    if (!h)
        return (int)cudaErrorInvalidValue;
    if (n_origins == 0 || n_lags == 0)
        return 0;
    if (!rho || !out || K == 0)
        return (int)cudaErrorInvalidValue;
    const unsigned long long n = (unsigned long long)n_origins * n_lags;
    k_fkt<<<(unsigned int)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(rho, T, K, n_origins, n_lags, out);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
    }

// ---- F(k,t) tracker: rho(t) and its correlation with every stored reference, on the device, each step ----------------
static uint64_t fkt_words(const cavb200_handle* h) { return 2ull + h->fkt_max_refs + 2ull * h->fkt_K; }
static double* fkt_kvec(cavb200_handle* h) { return h->fkt_track; }
static double* fkt_rho(cavb200_handle* h) { return h->fkt_track + 3ull * h->fkt_K; }
static double* fkt_refs(cavb200_handle* h) { return fkt_rho(h) + 2ull * h->fkt_K; }
static double* fkt_ring(cavb200_handle* h) { return fkt_refs(h) + 2ull * h->fkt_K * h->fkt_max_refs; }
static unsigned long long* fkt_counter(cavb200_handle* h)
    {
    return reinterpret_cast<unsigned long long*>(fkt_ring(h) + h->fkt_capacity * fkt_words(h));
    }

void cavb_fkt_track_release(cavb200_handle* h)
    {
    cudaFree(h->fkt_track);
    h->fkt_track = nullptr;
    h->fkt_K = h->fkt_max_refs = h->fkt_n_refs = 0;
    h->fkt_capacity = 0;
    }

extern "C" int cavb200_fkt_track_open(cavb200_handle* h, const double* kvec_host, uint32_t K, uint32_t max_references,
                                      uint32_t capacity, uint32_t N)
    {
    if (!h || !kvec_host || K == 0 || max_references == 0 || max_references > 1024 || capacity == 0)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaSetDevice(h->device));
    cavb_fkt_track_release(h);
    const uint64_t words = 2ull + max_references + 2ull * K;
    const size_t bytes = sizeof(double) * (5ull * K + 2ull * K * max_references + (uint64_t)capacity * words) +
                         sizeof(unsigned long long);
    double* buf = nullptr;
    CAVB_CHECK(cudaMalloc((void**)&buf, bytes));
    h->fkt_track = buf;
    h->fkt_K = K;
    h->fkt_max_refs = max_references;
    h->fkt_capacity = capacity;
    int err = (int)cudaMemset(buf, 0, bytes);
    if (!err)
        err = (int)cudaMemcpy(fkt_kvec(h), kvec_host, sizeof(double) * 3ull * K, cudaMemcpyHostToDevice);
    // the table, the kernels' attributes and the slice workspace now, so that a step never synchronises
    if (!err)
        err = rhok_prime(h, N, K);
    if (err)
        cavb_fkt_track_release(h);
    return err;
    }

extern "C" int cavb200_fkt_track_step(cavb200_handle* h, const double* pos, uint32_t N, uint64_t timestep, uint32_t flags,
                                      void* stream)
    {
    if (!h || !h->fkt_track || flags == 0 || (flags & ~(CAVB200_FKT_RECORD | CAVB200_FKT_ADD_REFERENCE)))
        return (int)cudaErrorInvalidValue;
    if ((flags & CAVB200_FKT_ADD_REFERENCE) && h->fkt_n_refs >= h->fkt_max_refs)
        return (int)cudaErrorInvalidValue;
    const uint32_t K = h->fkt_K;
    // rho(t) into the slot: the cavb200_rhok launch for one Scalar4 frame (its checks: NULL pos with N > 0, alignment)
    const int err = rhok_launch(h, pos, 4, 4ull * N, N, 1, fkt_kvec(h), K, fkt_rho(h), stream);
    if (err)
        return err;
    cudaLaunchAttribute pdl_attr;
    pdl_attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl_attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    // one thread per reference (at most 1024), and at least 256 for the copies of rho
    const uint32_t threads = h->fkt_max_refs <= 256 ? 256u : (h->fkt_max_refs + 31u) / 32u * 32u;
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(threads);
    cfg.stream = (cudaStream_t)stream;
    cfg.attrs = &pdl_attr;
    cfg.numAttrs = h->tune.pdl ? 1 : 0;
    const double* rho = fkt_rho(h);
    double* refs = fkt_refs(h);
    uint32_t max_refs = h->fkt_max_refs, n_refs = h->fkt_n_refs;
    double ts = (double)timestep;
    double* ring = fkt_ring(h);
    unsigned long long* count = fkt_counter(h);
    unsigned long long cap = h->fkt_capacity;
    void* args[] = {(void*)&rho, (void*)&refs, (void*)&K,  (void*)&max_refs, (void*)&n_refs,
                    (void*)&flags, (void*)&ts, (void*)&ring, (void*)&count,    (void*)&cap};
    CAVB_CHECK(cudaLaunchKernelExC(&cfg, (const void*)k_fkt_track, args));
    h->launches += 1;
    if (flags & CAVB200_FKT_ADD_REFERENCE)
        h->fkt_n_refs += 1;
    return 0;
    }

extern "C" int cavb200_fkt_track_read(cavb200_handle* h, double* out, uint32_t max_records, uint32_t* n_out,
                                      uint64_t* total, void* stream)
    {
    if (!h || !h->fkt_track || (!out && max_records) || !n_out)
        return (int)cudaErrorInvalidValue;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long cnt = 0;
    CAVB_CHECK(cudaMemcpyAsync(&cnt, fkt_counter(h), sizeof(cnt), cudaMemcpyDeviceToHost, s));
    CAVB_CHECK(cudaStreamSynchronize(s));
    const unsigned long long cap = h->fkt_capacity;
    const uint64_t words = fkt_words(h);
    unsigned long long have = cnt < cap ? cnt : cap; // records still in the ring
    if (have > max_records)
        have = max_records;
    // the newest `have` records, oldest first; the ring wraps at most once inside that span
    const unsigned long long first = cnt - have;
    unsigned long long done = 0;
    while (done < have)
        {
        const unsigned long long at = (first + done) % cap;
        unsigned long long run = cap - at;
        if (run > have - done)
            run = have - done;
        CAVB_CHECK(cudaMemcpyAsync(out + done * words, fkt_ring(h) + at * words, run * words * sizeof(double),
                                   cudaMemcpyDeviceToHost, s));
        done += run;
        }
    CAVB_CHECK(cudaStreamSynchronize(s));
    *n_out = (uint32_t)have;
    if (total)
        *total = cnt;
    return 0;
    }
