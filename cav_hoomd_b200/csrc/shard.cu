// shard.cu -- particle-sharded multi-GPU step (one process per GPU).
//
// New functionality relative to the reference (which sums the dipole over the local getN() only
// and never reduces across ranks, src/CavityForceCompute.cc:142,166; SURVEY.md 2.3): each rank
// owns a contiguous block of particles and one 128-byte record per rank crosses NVLink per step:
//   kernel A  reduce over the local particles; the last CTA merges the CTA records into the
//             rank's record {d as (hi,lo) pairs, sum m|v|^2, first 'L' (global index, q, term), n_L}
//   exchange  mode 0: ncclAllGather (libnccl resolved with dlopen, no link-time dependency)
//             mode 1: the same last CTA stores the record straight into every peer's mailbox
//                     (CUDA-IPC mapped peer memory over NVLink) and then raises a sequence flag;
//                     there is no collective call and no host involvement
//   kernel B  every CTA merges the nranks records in RANK ORDER (deterministic, identical on all
//             ranks), forms Dq / F_L / energies / alpha, and applies forces and the rescale.
//             In mode 1 it first spins (bounded) on its own flags.
// Because d travels as compensated pairs the result differs from the single-GPU one only in the
// final rounding of hi+lo.
#include "hotpath.cuh"

#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <string.h>

namespace cavb
    {
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v)
    {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
    }
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p)
    {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
    }

// mailbox of a rank: [kind: 0 two-kernel path / split dipole, 1 split KE][parity][16 ranks] records
constexpr int MAILBOX_RECORDS = 64;
constexpr unsigned long long SHARD_EPOCH_TAG = 1ull << 62; // keeps shard epochs apart from the single-GPU counter

struct PeerTable
    {
    Partial* mailbox[16];
    unsigned long long* flags[16];
    };

// kernel A
template<int UNROLL, int LB>
__global__ void __launch_bounds__(LB, LB == 384 ? 2 : 1)
    k_shard_reduce(ForceIn f, BussiIn b, Partial* recs, unsigned long long* ticket, Partial* rank_record, int mode,
                   int rank, int nranks, unsigned long long seq, PeerTable peers)
    {
    __shared__ BlockScratch sc;
    __shared__ int s_last;
    if (threadIdx.x == 0)
        sc.flags = 0u;
    reduce_phase<true, true, UNROLL>(f, b, sc);
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
    combine_phase<true, true, false, false>(recs, (int)gridDim.x, 0ull, f, b, sc, nullptr, false);
    if (threadIdx.x == 0)
        *ticket = 0ull;
    if (mode == 0)
        {
        if (threadIdx.x == 0)
            publish_record(rank_record, sc.rec, 0ull); // ncclAllGather sends it from here
        return;
        }
    // mode 1: thread `peer` stores the five sectors into that peer's mailbox, then one flag per peer
    const int parity = (int)(seq & 1ull);
    if ((int)threadIdx.x < nranks)
        publish_record(peers.mailbox[threadIdx.x] + (size_t)parity * 16 + rank, sc.rec, 0ull);
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < nranks)
        st_release_sys_u64(peers.flags[threadIdx.x] + rank, seq);
    }

// kernel B
template<int UNROLL, int LB>
__global__ void __launch_bounds__(LB, LB == 384 ? 2 : 1)
    k_shard_apply(ForceIn f, BussiIn b, const Partial* gathered, Scalars* scalars, int mode, int nranks,
                  unsigned long long seq, const unsigned long long* my_flags)
    {
    __shared__ BlockScratch sc;
    __shared__ int s_timeout;
    if (threadIdx.x == 0)
        {
        s_timeout = 0;
        sc.flags = 0u;
        }
    __syncthreads();
    if (mode == 1 && (int)threadIdx.x < nranks)
        {
        const unsigned long long t0 = globaltimer_ns();
        while (ld_acquire_sys_u64(my_flags + threadIdx.x) < seq)
            {
            if (globaltimer_ns() - t0 > 2000000000ull) // 2 s (peers may start late): never hang the GPU
                {
                s_timeout = 1;
                break;
                }
            }
        }
    __syncthreads();
    if (threadIdx.x == 0 && s_timeout)
        sc.flags = 1u;
    const Partial* recs = gathered + (mode == 1 ? (size_t)(seq & 1ull) * 16 : 0);
    combine_phase<true, true, false, true>(recs, nranks, 0ull, f, b, sc, scalars, blockIdx.x == 0);
    if (sc.fin.timeout)
        return;
    apply_phase<true, true, UNROLL>(sc.fin, f, b);
    }

// ---- ONE kernel per rank and step (mode 1, default) ----------------------------------------------
// The split-phase schedule of k_split with the NVLink exchange inside it:
//   dipole reduce -> CTA records -> CTA 0 folds them into the rank's record and stores it straight
//   into every peer's mailbox (peer memory, one 32-byte sector per store, self-validating with the
//   step number -- no flag, no fence, no collective call, no second launch);
//   KE reduce -> the same for the kinetic energy;
//   every CTA then folds the nranks dipole records that arrived in ITS OWN GPU's mailbox (rank order,
//   so every CTA of every rank forms bit-identical Dq) and writes forces; the KE records have crossed
//   NVLink in the meantime: alpha, rescale.
// Each exchange therefore has a whole streaming pass to complete behind.
template<int UNROLL, int LB>
__global__ void __launch_bounds__(LB, LB == 384 ? 2 : 1)
    k_shard_split(ForceIn f, BussiIn b, Partial* recsF, Partial* recsB, Scalars* scalars, const Partial* my_mailbox,
                  int rank, int nranks, unsigned long long seq, PeerTable peers)
    {
    __shared__ BlockScratch sc;
    const unsigned long long epoch = seq | SHARD_EPOCH_TAG;
    const size_t slot = (size_t)(seq & 1ull) * 16;
    // programmatic dependent launch (as the single-GPU kernels, hotpath.cu): nothing below may touch global memory before
    // the previous kernel of the stream has completed
    pdl_wait();
    if (threadIdx.x == 0)
        sc.flags = 0u;
    reduce_phase<true, false, UNROLL>(f, b, sc);
    if (threadIdx.x == 0)
        publish_record(recsF + blockIdx.x, sc.rec, epoch);
    if (blockIdx.x == 0)
        {
        combine_phase<true, false, true, false>(recsF, (int)gridDim.x, epoch, f, b, sc, nullptr, false);
        if ((int)threadIdx.x < nranks)
            publish_record(peers.mailbox[threadIdx.x] + slot + rank, sc.rec, epoch);
        __syncthreads(); // sc.rec is rewritten by the next block merge
        }
    reduce_phase<false, true, UNROLL>(f, b, sc);
    if (threadIdx.x == 0)
        publish_record(recsB + blockIdx.x, sc.rec, epoch);
    if (blockIdx.x == 0)
        {
        combine_phase<false, true, true, false>(recsB, (int)gridDim.x, epoch, f, b, sc, nullptr, false);
        if ((int)threadIdx.x < nranks)
            publish_record(peers.mailbox[threadIdx.x] + 32 + slot + rank, sc.rec, epoch);
        __syncthreads();
        }
    combine_phase<true, false, true, true, true>(my_mailbox + slot, nranks, epoch, f, b, sc, scalars, blockIdx.x == 0);
    const bool timeout_f = sc.fin.timeout != 0;
    if (!timeout_f)
        apply_phase<true, false, UNROLL>(sc.fin, f, b);
    __syncthreads();
    combine_phase<false, true, true, true, true>(my_mailbox + 32 + slot, nranks, epoch, f, b, sc, scalars, blockIdx.x == 0);
    if (sc.fin.timeout || timeout_f)
        {
        if (threadIdx.x == 0)
            raise_fault(scalars); // a record never arrived: outputs not (all) written, counted in cavb200_fault_count
        return;
        }
    pdl_launch_dependents(); // the next kernel's CTAs may take the SMs this grid's CTAs leave
    apply_phase<false, true, UNROLL>(sc.fin, f, b);
    }

// (A folder-CTA version of this kernel, as k_split_folder in hotpath.cu, was measured at 2 x 2M particles:
// 63.1 vs 63.5 us per step, with one 76 us outlier -- the rank-level folds already hide behind the long
// streaming passes of a 2M-particle shard.  Dropped.)

// ---- NCCL through dlopen ----------------------------------------------------------------------
struct NcclApi
    {
    void* lib;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    };

static NcclApi* nccl_api()
    {
    static NcclApi api = {};
    static int tried = 0;
    if (!tried)
        {
        tried = 1;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (int i = 0; i < 2 && !api.lib; i++)
            api.lib = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (api.lib)
            {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
            api.AllGather = (decltype(api.AllGather))dlsym(api.lib, "ncclAllGather");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
            if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.CommDestroy)
                api.lib = nullptr;
            }
        }
    return api.lib ? &api : nullptr;
    }

static int ensure_mailbox(cavb200_handle* h)
    {
    ShardState& sh = h->shard;
    if (sh.mailbox_alloc)
        return 0;
    // [2 parities][16 ranks] records + [16] flags, zeroed
    const size_t bytes = sizeof(Partial) * MAILBOX_RECORDS + sizeof(unsigned long long) * 16;
    CAVB_CHECK(cudaMalloc(&sh.mailbox_alloc, bytes));
    CAVB_CHECK(cudaMemset(sh.mailbox_alloc, 0, bytes));
    sh.gather = reinterpret_cast<Partial*>(sh.mailbox_alloc);
    sh.flags = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(sh.mailbox_alloc) + sizeof(Partial) * MAILBOX_RECORDS);
    sh.peer_mailbox[0] = sh.gather;
    sh.peer_flags[0] = sh.flags;
    return 0;
    }

template<int UNROLL, int LB> static int launch_shard_t(cavb200_handle* h, const ForceIn& f, const BussiIn& b, cudaStream_t s)
    {
    ShardState& sh = h->shard;
    int rc = ensure_mailbox(h);
    if (rc)
        return rc;
    const int threads = h->tune.threads > LB ? LB : h->tune.threads;
    const unsigned long long work = f.N > b.n ? f.N : b.n;
    unsigned long long want = (work + threads - 1) / threads;
    if (want < 1)
        want = 1;
    int max_grid = h->num_sms * h->tune.ctas_per_sm;
    if (max_grid > MAX_PARTIALS)
        max_grid = MAX_PARTIALS;
    const int grid = (int)(want < (unsigned long long)max_grid ? want : (unsigned long long)max_grid);
    sh.seq += 1;
    PeerTable peers;
    for (int r = 0; r < 16; r++)
        {
        peers.mailbox[r] = sh.peer_mailbox[r];
        peers.flags[r] = sh.peer_flags[r];
        }
    const int nranks = sh.nranks < 1 ? 1 : sh.nranks;
    const int mode = (nranks == 1 && sh.mode == 0) ? 1 : sh.mode; // one rank: the mailbox path is local
    if (nranks == 1)
        {
        peers.mailbox[0] = sh.gather;
        peers.flags[0] = sh.flags;
        }
    if (mode == 1 && h->tune.variant >= 1 && b.rescale)
        {
        // single persistent kernel: the CTAs wait on each other's records, so the grid must be co-resident
        int per_sm = 0;
        CAVB_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_shard_split<UNROLL, LB>, threads, 0));
        if (per_sm < 1)
            return (int)cudaErrorLaunchOutOfResources;
        int g = grid;
        if (g > per_sm * h->num_sms)
            g = per_sm * h->num_sms;
        if (g > MAX_PARTIALS / 2)
            g = MAX_PARTIALS / 2;
        ForceIn ff = f;
        BussiIn bb = b;
        Partial *recsF = h->partials, *recsB = h->partials + MAX_PARTIALS / 2;
        Scalars* sca = h->scalars;
        const Partial* box = sh.gather;
        int rank = sh.rank, nr = nranks;
        unsigned long long seq = sh.seq;
        void* args[] = {&ff, &bb, &recsF, &recsB, &sca, &box, &rank, &nr, &seq, &peers};
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(g);
        cfg.blockDim = dim3(threads);
        cfg.stream = s;
        // as hotpath.cu: programmatic dependent launch, or -- tuning pdl=0 -- the cooperative attribute, with which the
        // driver itself refuses a grid that cannot be co-resident
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
        CAVB_CHECK(cudaLaunchKernelExC(&cfg, (const void*)k_shard_split<UNROLL, LB>, args));
        h->launches += 1;
        return 0;
        }
    Partial* rank_record = h->partials + MAX_PARTIALS - 1;
    k_shard_reduce<UNROLL, LB><<<grid, threads, 0, s>>>(f, b, h->partials, h->counters + 4, rank_record, mode, sh.rank, nranks,
                                                     sh.seq, peers);
    CAVB_CHECK(cudaGetLastError());
    if (mode == 0)
        {
        NcclApi* api = nccl_api();
        if (!api || !sh.nccl_comm)
            return (int)cudaErrorNotReady;
        if (api->AllGather(rank_record, sh.gather, sizeof(Partial), ncclChar, (ncclComm_t)sh.nccl_comm, s) != ncclSuccess)
            return (int)cudaErrorUnknown;
        }
    k_shard_apply<UNROLL, LB><<<grid, threads, 0, s>>>(f, b, sh.gather, h->scalars, mode, nranks, sh.seq, sh.flags);
    CAVB_CHECK(cudaGetLastError());
    h->launches += 2;
    return 0;
    }

int launch_shard_step(cavb200_handle* h, const ForceIn* f, const BussiIn* b, cudaStream_t s)
    {
    switch (h->tune.unroll)
        {
    case 8:
        return launch_shard_t<8, 256>(h, *f, *b, s);
    case 4:
        return launch_shard_t<4, 512>(h, *f, *b, s);
    default:
        if (h->tune.threads <= 384)
            return launch_shard_t<2, 384>(h, *f, *b, s);
        return launch_shard_t<2, 1024>(h, *f, *b, s);
        }
    }
    } // namespace cavb

using namespace cavb;

void cavb_shard_release(cavb200_handle* h)
    {
    ShardState& sh = h->shard;
    for (int r = 0; r < 16; r++)
        if (r != sh.rank && sh.peer_mailbox[r] && sh.nranks > 1)
            cudaIpcCloseMemHandle(sh.peer_mailbox[r]);
    if (sh.nccl_comm)
        {
        NcclApi* api = nccl_api();
        if (api)
            api->CommDestroy((ncclComm_t)sh.nccl_comm);
        }
    cudaFree(sh.mailbox_alloc);
    memset(&sh, 0, sizeof(sh));
    }

extern "C"
    {
int cavb200_shard_nccl_unique_id(void* out128)
    {
    if (!out128)
        return (int)cudaErrorInvalidValue;
    NcclApi* api = nccl_api();
    if (!api)
        return (int)cudaErrorSharedObjectInitFailed;
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == CAVB200_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
    if (api->GetUniqueId(&id) != ncclSuccess)
        return (int)cudaErrorUnknown;
    memcpy(out128, &id, sizeof(id));
    return 0;
    }

int cavb200_shard_init_nccl(cavb200_handle* h, const void* unique_id128, int rank, int nranks)
    {
    if (!h || !unique_id128 || nranks < 1 || nranks > 16 || rank < 0 || rank >= nranks)
        return (int)cudaErrorInvalidValue;
    NcclApi* api = nccl_api();
    if (!api)
        return (int)cudaErrorSharedObjectInitFailed;
    CAVB_CHECK(cudaSetDevice(h->device));
    int rc = ensure_mailbox(h);
    if (rc)
        return rc;
    ncclUniqueId id;
    memcpy(&id, unique_id128, sizeof(id));
    ncclComm_t comm;
    if (api->CommInitRank(&comm, nranks, id, rank) != ncclSuccess)
        return (int)cudaErrorUnknown;
    h->shard.nccl_comm = comm;
    h->shard.rank = rank;
    h->shard.nranks = nranks;
    h->shard.mode = 0;
    return 0;
    }

int cavb200_shard_mailbox_export(cavb200_handle* h, void* out64)
    {
    if (!h || !out64)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaSetDevice(h->device));
    int rc = ensure_mailbox(h);
    if (rc)
        return rc;
    cudaIpcMemHandle_t mh;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    CAVB_CHECK(cudaIpcGetMemHandle(&mh, h->shard.mailbox_alloc));
    memcpy(out64, &mh, sizeof(mh));
    return 0;
    }

int cavb200_shard_mailbox_open(cavb200_handle* h, const void* handles, int rank, int nranks)
    {
    if (!h || !handles || nranks < 1 || nranks > 16 || rank < 0 || rank >= nranks)
        return (int)cudaErrorInvalidValue;
    CAVB_CHECK(cudaSetDevice(h->device));
    int rc = ensure_mailbox(h);
    if (rc)
        return rc;
    ShardState& sh = h->shard;
    for (int r = 0; r < nranks; r++)
        {
        void* base = nullptr;
        if (r == rank)
            base = sh.mailbox_alloc;
        else
            {
            cudaIpcMemHandle_t mh;
            memcpy(&mh, (const char*)handles + 64 * r, sizeof(mh));
            CAVB_CHECK(cudaIpcOpenMemHandle(&base, mh, cudaIpcMemLazyEnablePeerAccess));
            }
        sh.peer_mailbox[r] = reinterpret_cast<Partial*>(base);
        sh.peer_flags[r] = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(base) + sizeof(Partial) * MAILBOX_RECORDS);
        }
    sh.rank = rank;
    sh.nranks = nranks;
    sh.mode = 1;
    return 0;
    }

int cavb200_shard_set_mode(cavb200_handle* h, int mode)
    {
    if (!h || (mode != 0 && mode != 1))
        return (int)cudaErrorInvalidValue;
    if (mode == 0 && h->shard.nranks > 1 && !h->shard.nccl_comm)
        return (int)cudaErrorNotReady;
    if (mode == 1 && h->shard.nranks > 1 && !h->shard.peer_mailbox[(h->shard.rank + 1) % h->shard.nranks])
        return (int)cudaErrorNotReady;
    h->shard.mode = mode;
    return 0;
    }

int cavb200_shard_step(cavb200_handle* h, const double* pos, const double* charge, const int32_t* image, double* force,
                       double* vel, uint32_t N_local, uint64_t index_offset, double Lx, double Ly, double Lz,
                       uint32_t L_typeid, const cavb200_params* params, uint32_t group_first, uint32_t n_group,
                       const cavb200_bussi_args* bussi, void* stream)
    {
    if (!h || !params || !bussi)
        return (int)cudaErrorInvalidValue;
    if ((unsigned long long)group_first + n_group > N_local)
        return (int)cudaErrorInvalidValue;
    // every rank must take part in the exchange even with an empty shard, so no N == 0 shortcut
    if (N_local > 0 && (!pos || !charge || !image || !force))
        return (int)cudaErrorInvalidValue;
    if (n_group > 0 && !vel)
        return (int)cudaErrorInvalidValue;
    if ((reinterpret_cast<uintptr_t>(pos) & 31) || (reinterpret_cast<uintptr_t>(force) & 31)
        || (reinterpret_cast<uintptr_t>(vel) & 31))
        return (int)cudaErrorMisalignedAddress;
    ForceIn f;
    f.pos = reinterpret_cast<const double4*>(pos);
    f.charge = charge;
    f.image = image;
    f.force = reinterpret_cast<double4*>(force);
    f.N = N_local;
    f.index_offset = index_offset;
    f.Lx = Lx;
    f.Ly = Ly;
    f.Lz = Lz;
    f.L_typeid = L_typeid;
    f.g = params->couplstr;
    f.K = params->K;
    fill_force_constants(f);
    BussiIn b;
    b.vel = reinterpret_cast<double4*>(vel);
    b.gidx = nullptr;
    b.first = group_first;
    b.n = n_group;
    b.rescale = bussi->deltaT != 0.0;
    b.stream_st = (uint64_t)n_group * 116ull > (63ull << 20); // as api.cu fill_bussi
    fill_bussi_constants(b, bussi);
    h->index_offset = index_offset;
    return launch_shard_step(h, &f, &b, (cudaStream_t)stream);
    }
    }
