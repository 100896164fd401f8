/*
 * pom_batch.cu — implementation of the C ABI in include/pom_batch.h (libpom_b200.so).
 *
 * Host side of the product: owns device memory, streams and launches; every simulation step runs
 * in the sm_100a kernels of pom_kernels.cuh.  There is deliberately no host stepping path here:
 * without a CUDA device every entry point fails with POM_E_CUDA.
 */
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sched.h>
#include <string>
#include <vector>
#include <new>

#include "pom_batch.h"
#include "pom_kernels.cuh"

namespace
{

thread_local std::string g_err;

int fail(int code, const char* what, cudaError_t ce = cudaSuccess)
{
    g_err = what;
    if(ce != cudaSuccess)
    {
        g_err += ": ";
        g_err += cudaGetErrorString(ce);
    }
    return code;
}

/* temporary device allocation, released on every return path */
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if(p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes); }
    template<typename T> T* as() const { return static_cast<T*>(p); }
};

#define CK(expr) do { cudaError_t ce_ = (expr); if(ce_ != cudaSuccess) return fail(POM_E_CUDA, #expr, ce_); } while(0)

/* The record array in compressible device memory.  Each tick streams the whole array through DRAM, and most of a
 * record's bytes are zero (empty board cells, unused bomb and flame ring slots, the pad bytes): with generic compression
 * the hardware moves fewer DRAM bytes for the same lines, losslessly and unseen by the kernels.  Compressible memory
 * exists only through the driver's virtual memory API; its entry points are looked up at run time, so the library
 * links against the runtime alone. */
struct Driver {
    PFN_cuDeviceGet_v2000 DeviceGet = nullptr;
    PFN_cuDeviceGetAttribute_v2000 DeviceGetAttribute = nullptr;
    PFN_cuMemGetAllocationGranularity_v10020 MemGetAllocationGranularity = nullptr;
    PFN_cuMemCreate_v10020 MemCreate = nullptr;
    PFN_cuMemGetAllocationPropertiesFromHandle_v10020 MemGetAllocationPropertiesFromHandle = nullptr;
    PFN_cuMemAddressReserve_v10020 MemAddressReserve = nullptr;
    PFN_cuMemMap_v10020 MemMap = nullptr;
    PFN_cuMemSetAccess_v10020 MemSetAccess = nullptr;
    PFN_cuMemUnmap_v10020 MemUnmap = nullptr;
    PFN_cuMemRelease_v10020 MemRelease = nullptr;
    PFN_cuMemAddressFree_v10020 MemAddressFree = nullptr;
    bool ok = false;
};

template<typename F>
bool entry(const char* name, F* fn)
{
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if(cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
    {
        cudaGetLastError();
        return false;
    }
    *fn = reinterpret_cast<F>(p);
    return true;
}

const Driver& driver()
{
    static const Driver d = [] {
        Driver x;
        x.ok = entry("cuDeviceGet", &x.DeviceGet) && entry("cuDeviceGetAttribute", &x.DeviceGetAttribute) &&
               entry("cuMemGetAllocationGranularity", &x.MemGetAllocationGranularity) && entry("cuMemCreate", &x.MemCreate) &&
               entry("cuMemGetAllocationPropertiesFromHandle", &x.MemGetAllocationPropertiesFromHandle) &&
               entry("cuMemAddressReserve", &x.MemAddressReserve) && entry("cuMemMap", &x.MemMap) &&
               entry("cuMemSetAccess", &x.MemSetAccess) && entry("cuMemUnmap", &x.MemUnmap) &&
               entry("cuMemRelease", &x.MemRelease) && entry("cuMemAddressFree", &x.MemAddressFree);
        return x;
    }();
    return d;
}

/* Maps `bytes` (rounded up to the allocation granularity) of compressible memory on `device`; returns the mapped size, or
 * 0 when the device, the driver or the grant says no.  The driver may hand out uncompressible memory for a compressible
 * request: the granted properties are read back and such memory is given back. */
size_t map_compressible(int device, size_t bytes, void** out)
{
    const Driver& d = driver();
    if(!d.ok) return 0;
    CUdevice dev = 0;
    int vmm = 0, comp = 0;
    if(d.DeviceGet(&dev, device) != CUDA_SUCCESS ||
       d.DeviceGetAttribute(&vmm, CU_DEVICE_ATTRIBUTE_VIRTUAL_MEMORY_MANAGEMENT_SUPPORTED, dev) != CUDA_SUCCESS || !vmm ||
       d.DeviceGetAttribute(&comp, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev) != CUDA_SUCCESS || !comp)
        return 0;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = dev;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if(d.MemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM) != CUDA_SUCCESS || gran == 0) return 0;
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h = 0;
    if(d.MemCreate(&h, size, &prop, 0) != CUDA_SUCCESS) return 0;
    CUmemAllocationProp got = {};
    CUdeviceptr va = 0;
    CUmemAccessDesc access = {};
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    const bool granted = d.MemGetAllocationPropertiesFromHandle(&got, h) == CUDA_SUCCESS &&
                         got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
    const bool reserved = granted && d.MemAddressReserve(&va, size, gran, 0, 0) == CUDA_SUCCESS;
    const bool mapped = reserved && d.MemMap(va, size, 0, h, 0) == CUDA_SUCCESS;
    const bool ok = mapped && d.MemSetAccess(va, size, &access, 1) == CUDA_SUCCESS;
    d.MemRelease(h);                           /* from here on the mapping alone holds the memory */
    if(!ok)
    {
        if(mapped) d.MemUnmap(va, size);
        if(reserved) d.MemAddressFree(va, size);
        return 0;
    }
    *out = reinterpret_cast<void*>(va);
    return size;
}

/* the handle's record array: compressible memory where the device grants it, cudaMalloc otherwise.  *mapped is the
 * compressible mapping's size, 0 for cudaMalloc: it selects how free_records gives the memory back.
 * Only the records: pom_device_alloc (the bench's move ring, observation slabs) and the template pool in compressible
 * memory as well measured within 0.1 % of this on every leg of bench.py (B200, profiles/bench_compressible.jsonl), so
 * they stay on cudaMalloc. */
cudaError_t alloc_records(int device, size_t bytes, uint8_t** out, size_t* mapped)
{
    void* p = nullptr;
    *mapped = map_compressible(device, bytes, &p);
    if(*mapped) { *out = static_cast<uint8_t*>(p); return cudaSuccess; }
    return cudaMalloc(reinterpret_cast<void**>(out), bytes);
}

void free_records(uint8_t* p, size_t mapped)
{
    if(!p) return;
    if(!mapped) { cudaFree(p); return; }
    /* cudaFree waits for the device before it frees; an unmap is given the same wait, so that no kernel of any handle
     * on this device (an expansion reading these records into another handle) still uses the range */
    cudaDeviceSynchronize();
    const Driver& d = driver();
    d.MemUnmap(reinterpret_cast<CUdeviceptr>(p), mapped);
    d.MemAddressFree(reinterpret_cast<CUdeviceptr>(p), mapped);
}

constexpr uint64_t TILE_ALIGN = 256;           /* records are allocated in whole tiles of the largest TPB */
constexpr uint64_t XFER_CHUNK = 65536;         /* envs per AoS staging chunk (66 MB)                      */
constexpr size_t   FLUSH_BYTES = size_t(256) << 20;

}

struct pom_batch {
    int       device = 0;
    uint64_t  n_envs = 0;
    uint64_t  n_alloc = 0;                     /* n_envs rounded up to TILE_ALIGN */
    uint64_t  env_offset = 0;
    uint32_t  n_templates = 0;
    uint32_t  max_ticks = 0;
    int       tpb = 128;
    int       n_sms = 1;
    int       ws_nw = 20;
    uint32_t  attr_ws = 0;
    uint32_t  walk = 0;                        /* whole-batch per-tick launches so far: odd ones walk the batch backwards (StepIO::reverse) */
    int       pingpong = 1;                    /* POM_STEP_PINGPONG=0 switches the alternation off (experiments) */
    int       no_spec = 0;                     /* POM_WS_NOSPEC=1: always the generic image of k_step_ws / k_rollout */
    int       policy_pertick = 1;              /* POM_ROLL_POLICY=fused: pom_batch_rollout with SimpleAgents always uses the fused kernel */
    int       obs_fused = 0;                   /* POM_OBS_FUSED=1: pom_batch_step_observe / pom_step_compact_io::obs_dev write the planes
                                                  from inside the step kernel instead of launching k_observe_planes behind it */
    int       step_kernel = 0;                 /* 0 = k_step_ws (persistent, warp-specialised), 1 = k_step (one CTA per tile); POM_STEP_KERNEL=tile */
    int       step_parts = 2;                  /* POM_STEP_PARTS=2..16: launches per pom_batch_step with POM_STEP_OVERLAP */
    int       chunks = 6;                      /* POM_CHUNKS=1..MAX_CHUNKS: chunks of pom_batch_step_host's copy pipeline */
    int       zerocopy = 1;                    /* POM_ZEROCOPY=0: pom_batch_step_host takes the copy pipeline for pinned buffers too */
    bool      teams = false;                   /* POM_INIT_TEAMS: the 2v2 team game, fixed for the handle's life; every stepping or
                                                  acting launch takes the kernel images of this mode (POM_DISPATCH_MODE) */
    bool      radio = false;                   /* POM_INIT_RADIO (team game only, fixed for the handle's life): the records' radio bytes
                                                  hold the team messages; the observation planes take the RADIO images */
    int       policy_view = -1;                /* pom_batch_set_policy_view: >= 0 = the device SimpleAgent plays under fog of war
                                                  with this view (the FOG images, POM_DISPATCH_POLICY), < 0 = on the full state */
    uint8_t*  recs = nullptr;
    size_t    recs_mapped = 0;                 /* bytes of compressible memory mapped for recs (alloc_records); 0 = cudaMalloc */
    uint8_t*  templates = nullptr;
    uint32_t* episodes = nullptr;
    unsigned long long* stats = nullptr;
    uint32_t* moves_buf = nullptr;             /* n_envs x 4 bytes, for pom_batch_step_host */
    uint8_t*  status_buf = nullptr;            /* n_envs bytes                               */
    pom_state* aos_stage = nullptr;            /* XFER_CHUNK states                          */
    uint8_t*  st_stage = nullptr;
    uint32_t* bad_count = nullptr;
    uint32_t* fin_counter = nullptr;           /* device word behind the finished-env list of pom_batch_step_compact */
    uint32_t* policy = nullptr;                /* 9 x n_alloc words: SimpleAgent memories (allocated on first use) */
    void*     flush_buf = nullptr;
    uint32_t* idx_buf = nullptr;               /* root / source indices of pom_batch_expand_step on the device (grow-only) */
    uint64_t  idx_cap = 0;
    cudaEvent_t ev_expand = nullptr;           /* end of the last expansion INTO this handle: the source handle's stream waits for it */
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2] = { nullptr, nullptr };
    /* pom_batch_step_host pipelines chunks of the batch: H2D of chunk c+1 and D2H of chunk c-1 overlap the
     * kernel of chunk c (copy engines + SMs), ordered by events */
    static constexpr int MAX_CHUNKS = 16;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr, s_k2 = nullptr;   /* s_k2: second compute stream, so that the tail of one chunk's kernel overlaps the head of the next */
    cudaEvent_t ev_k2 = nullptr;
    cudaEvent_t ev_in[MAX_CHUNKS] = {}, ev_done[MAX_CHUNKS] = {}, ev_out = nullptr, ev_begin = nullptr;
    std::vector<int32_t> seeds;
    uint64_t  launches = 0;
    bool      forked = false;                  /* work is pending on s_k2 that the handle's stream has not waited for */
    uint64_t  attr_done = 0;                   /* kernels whose shared-memory attribute has been set on this handle's device */

    pomk::BatchParams params() const
    {
        pomk::BatchParams P;
        P.recs = recs; P.n_envs = n_envs; P.env_offset = env_offset; P.templates = templates;
        P.n_templates = n_templates; P.max_ticks = max_ticks;
        P.tmpl_mask = (n_templates & (n_templates - 1u)) == 0u ? n_templates - 1u : 0u; P.episodes = episodes; P.stats = stats;
        P.policy = policy; P.policy_stride = n_alloc;
        return P;
    }
};

namespace
{

/* Every entry point starts here.  If the previous call was a pom_batch_step with POM_STEP_OVERLAP, the second half of
 * the batch may still be in flight on the second compute stream: make the handle's stream wait for it, so that
 * everything else stays ordered on that one stream. */
int use(const pom_batch* cb, bool join = true)
{
    if(!cb) return fail(POM_E_ARG, "null handle");
    CK(cudaSetDevice(cb->device));
    pom_batch* b = const_cast<pom_batch*>(cb);
    if(join && b->forked)
    {
        CK(cudaEventRecord(b->ev_k2, b->s_k2));
        CK(cudaStreamWaitEvent(b->stream, b->ev_k2, 0));
        b->forked = false;
    }
    return POM_OK;
}

/* The dynamic shared-memory limit of a kernel is a per-device attribute: remember it per handle (one handle = one
 * device), not in a process-wide flag, so that handles on other GPUs and other host threads set it for themselves. */
enum { ATTR_STEP = 1, ATTR_ROLLOUT = 2, ATTR_ROLLOUT_POLICY = 4, ATTR_POLICY_MOVES = 8, ATTR_EXPAND = 16, ATTR_OBS = 32, ATTR_ROLLOUT_SPEC = 64, ATTR_OBS_CROPPED = 128 };
/* the RADIO images of k_observe_planes take bits 32 and 33 */
constexpr uint64_t ATTR_OBS_RADIO = uint64_t(1) << 32, ATTR_OBS_CROPPED_RADIO = uint64_t(1) << 33;
/* the bit of a kernel's team image, and of its FOG image (bits 16..23 for free-for-all, 24..31 for the team game) */
constexpr uint32_t attr_bit(uint32_t which, bool teams, bool fog = false) { return (fog ? which << 16 : which) << (teams ? 8 : 0); }

/* the handle's policy view as the FOG images take it: in the spare bits of the agent mask or draw (pomk::POLICY_VIEW_SHIFT) */
uint32_t policy_view_bits(const pom_batch* b)
{
    return uint32_t(b->policy_view > 15 ? 15 : b->policy_view) << pomk::POLICY_VIEW_SHIFT;
}

template<typename K>
int set_smem(pom_batch* b, uint64_t which, K kernel, uint32_t bytes)
{
    if(b->attr_done & which) return POM_OK;
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
    b->attr_done |= which;
    return POM_OK;
}

int ensure_stage(pom_batch* b)
{
    if(!b->aos_stage)
    {
        CK(cudaMalloc(&b->aos_stage, XFER_CHUNK * sizeof(pom_state)));
        CK(cudaMalloc(&b->st_stage, XFER_CHUNK));
        CK(cudaMalloc(&b->bad_count, sizeof(uint32_t)));
    }
    return POM_OK;
}

int ensure_policy(pom_batch* b)
{
    if(!b->policy)
    {
        CK(cudaMalloc(&b->policy, 9 * b->n_alloc * sizeof(uint32_t)));
        CK(cudaMemsetAsync(b->policy, 0, 9 * b->n_alloc * sizeof(uint32_t), b->stream));
    }
    return POM_OK;
}

int fill_from_templates(pom_batch* b)
{
    const uint64_t words = b->n_envs * POM_REC_WORDS;
    pomk::k_fill_from_templates<<<unsigned((words + 255) / 256), 256, 0, b->stream>>>(b->params());
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

/* builds the template pool on the device: InitState for the first n clean seeds >= first_seed */
int build_templates_from_seeds(pom_batch* b, int32_t first_seed)
{
    const uint32_t n = b->n_templates;
    if(n > (1u << 24)) return fail(POM_E_ARG, "pom_batch_init: at most 2^24 templates");
    if(int64_t(first_seed) + 16 * int64_t(n) + 4096 > 0x7FFFFFFFll) return fail(POM_E_ARG, "pom_batch_init: first_seed too close to INT_MAX for this many templates");
    uint32_t ncand = uint32_t(n * 2.2) + 64;
    for(int attempt = 0; attempt < 6; attempt++, ncand *= 2)
    {
        DevBuf cand_b, dirty_b, pick_b;
        CK(cand_b.alloc(size_t(ncand) * POM_REC_BYTES));
        CK(dirty_b.alloc(ncand));
        uint8_t* cand = cand_b.as<uint8_t>(); uint8_t* dirty = dirty_b.as<uint8_t>();
        pomk::k_make_templates<<<(ncand + 63) / 64, 64, 0, b->stream>>>(cand, dirty, first_seed, ncand);
        b->launches++;
        CK(cudaGetLastError());
        std::vector<uint8_t> h(ncand);
        CK(cudaMemcpyAsync(h.data(), dirty, ncand, cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
        std::vector<uint32_t> idx;
        for(uint32_t i = 0; i < ncand && idx.size() < n; i++) if(!h[i]) idx.push_back(i);
        if(idx.size() == n)
        {
            CK(pick_b.alloc(n * sizeof(uint32_t)));
            uint32_t* pick = pick_b.as<uint32_t>();
            CK(cudaMemcpyAsync(pick, idx.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream));
            const uint64_t words = uint64_t(n) * POM_REC_WORDS;
            pomk::k_gather_records<<<unsigned((words + 255) / 256), 256, 0, b->stream>>>(
                reinterpret_cast<uint32_t*>(b->templates), reinterpret_cast<const uint32_t*>(cand), pick, n, 0);
            b->launches++;
            CK(cudaGetLastError());
            CK(cudaStreamSynchronize(b->stream));
            b->seeds.resize(n);
            for(uint32_t k = 0; k < n; k++) b->seeds[k] = first_seed + int32_t(idx[k]);
            return POM_OK;
        }
    }
    return fail(POM_E_ARG, "could not find enough clean seeds");
}

int pack_into(pom_batch* b, uint8_t* dst_recs, uint64_t first, uint64_t count, const pom_state* states, const uint8_t* status, uint32_t* bad_total)
{
    int rc = ensure_stage(b);
    if(rc) return rc;
    for(uint64_t done = 0; done < count; done += XFER_CHUNK)
    {
        const uint64_t c = count - done < XFER_CHUNK ? count - done : XFER_CHUNK;
        CK(cudaMemcpyAsync(b->aos_stage, states + done, c * sizeof(pom_state), cudaMemcpyHostToDevice, b->stream));
        if(status) CK(cudaMemcpyAsync(b->st_stage, status + done, c, cudaMemcpyHostToDevice, b->stream));
        CK(cudaMemsetAsync(b->bad_count, 0, sizeof(uint32_t), b->stream));
        pomk::k_pack<<<unsigned((c + 127) / 128), 128, 0, b->stream>>>(b->aos_stage, status ? b->st_stage : nullptr, dst_recs, first + done, c, b->bad_count);
        b->launches++;
        CK(cudaGetLastError());
        uint32_t bad = 0;
        CK(cudaMemcpyAsync(&bad, b->bad_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
        *bad_total += bad;
    }
    return POM_OK;
}

/* geometry of the persistent per-tick kernel (k_step_ws): compute warps and slice buffers per CTA (= per SM) */
constexpr int WS_NW = 20, WS_NBUF = 24;

template<int NW, bool OBS, bool FREEZE = false, bool SPEC = false, bool TEAMS = false, bool REWARDS = false, bool RADIO = false>
int launch_step_ws(pom_batch* b, const pomk::BatchParams& P, const pomk::StepIO& io, uint32_t flags, cudaStream_t on)
{
    typedef pomk::RingScratch<WS_NBUF> R;
    /* NW is even and >= 12; the team images (NW = WS_NW only) take bits 24..26, the REWARDS images bits 27..28, the RADIO
     * image bit 29 */
    const uint32_t bit = RADIO ? (1u << 29) :
                         REWARDS ? (1u << (TEAMS ? 28 : 27)) :
                         TEAMS ? (1u << (24 + (FREEZE ? 2 : (OBS ? 1 : 0)))) :
                         SPEC ? 2u : (FREEZE ? 1u : (1u << (NW + (OBS ? 1 : 0))));
    if(!(b->attr_ws & bit))
    {
        CK(cudaFuncSetAttribute(pomk::k_step_ws<NW, WS_NBUF, OBS, FREEZE, SPEC, TEAMS, REWARDS, RADIO>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(R::BYTES)));
        b->attr_ws |= bit;
    }
    const uint64_t n_slices = (P.n_envs + 31) / 32;
    const unsigned grid = unsigned(n_slices < uint64_t(b->n_sms) ? n_slices : uint64_t(b->n_sms));
    pomk::k_step_ws<NW, WS_NBUF, OBS, FREEZE, SPEC, TEAMS, REWARDS, RADIO><<<grid, (NW + 1) * 32, R::BYTES, on ? on : b->stream>>>(P, io, flags);
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

/* rewards: pom_batch_step_rewards, whose output travels in io.obs, so this is decided first; radio: pom_batch_step_radio
 * (rewards, if any, in io.obs, the messages in io.fin_status) */
int launch_step_io(pom_batch* b, const pomk::BatchParams& P, pomk::StepIO io, uint32_t flags, cudaStream_t on, bool rewards = false,
                   bool radio = false)
{
    io.bulk = (reinterpret_cast<uintptr_t>(io.moves) & 15u) == 0u ? 1u : 0u;   /* TMA needs 16-byte alignment */
    /* whole-batch launches alternate the direction of the walk (L2 reuse between ticks, see StepIO::reverse) */
    if(P.n_envs == b->n_envs && b->pingpong) io.reverse = (b->walk++) & 1u;
    /* the REWARDS and RADIO images exist for the default geometry and the generic image only (no SPEC, no POM_WS_NW variants);
     * the radio is a team-game feature */
    if(radio) return launch_step_ws<WS_NW, false, false, false, true, true, true>(b, P, io, flags, on);
    if(rewards)
    {
        if(b->teams) return launch_step_ws<WS_NW, false, false, false, true, true>(b, P, io, flags, on);
        return launch_step_ws<WS_NW, false, false, false, false, true>(b, P, io, flags, on);
    }
    if(b->teams)
    {
        /* the team game has the generic images of the default geometry only: no SPEC image, no POM_WS_NW variants */
        if(flags & pomk::STEP_FREEZE_TRUNCATED) return launch_step_ws<WS_NW, false, true, false, true>(b, P, io, flags, on);
        if(io.obs) return launch_step_ws<WS_NW, true, false, false, true>(b, P, io, flags, on);
        return launch_step_ws<WS_NW, false, false, false, true>(b, P, io, flags, on);
    }
    if(flags & pomk::STEP_FREEZE_TRUNCATED) return launch_step_ws<WS_NW, false, true>(b, P, io, flags, on);
    /* the specialised image (k_step_ws, SPEC) for the plain loop */
    if(b->ws_nw == WS_NW && (flags & ~uint32_t(POM_STEP_OVERLAP)) == uint32_t(POM_STEP_AUTORESET | POM_STEP_COUNT) && io.bulk &&
       !io.status_out && !io.obs && !io.joint && !io.done_bits && !io.fin_env && !b->no_spec)
        return launch_step_ws<WS_NW, false, false, true>(b, P, io, flags, on);
    if(io.obs) return launch_step_ws<WS_NW, true>(b, P, io, flags, on);
    /* persistent, warp-specialised: one CTA per SM; POM_WS_NW picks the number of compute warps (experiments) */
    switch(b->ws_nw)
    {
    case 12: return launch_step_ws<12, false>(b, P, io, flags, on);
    case 14: return launch_step_ws<14, false>(b, P, io, flags, on);
    case 16: return launch_step_ws<16, false>(b, P, io, flags, on);
    case 18: return launch_step_ws<18, false>(b, P, io, flags, on);
    case 22: return launch_step_ws<22, false>(b, P, io, flags, on);
    default: return launch_step_ws<WS_NW, false>(b, P, io, flags, on);
    }
}

template<int TPB, bool TEAMS = false>
int launch_step(pom_batch* b, const uint8_t* moves_dev, uint32_t flags, uint8_t* status_dev, uint64_t first = 0, uint64_t count = 0, cudaStream_t on = nullptr,
                bool tile_kernel = false)
{
    /* envs [first, first + count) only (first is a multiple of TPB); count == 0 means the whole batch */
    pomk::BatchParams P = b->params();
    if(count)
    {
        P.recs += first * POM_REC_BYTES; P.episodes += first; P.env_offset += first; P.n_envs = count;
        moves_dev += 4 * first;
        if(status_dev) status_dev += first;
    }
    if(b->step_kernel == 0 && !tile_kernel)
    {
        pomk::StepIO io{};
        io.moves = moves_dev;
        io.status_out = status_dev;
        return launch_step_io(b, P, io, flags, on);
    }
    { int rc = set_smem(b, attr_bit(ATTR_STEP, TEAMS), pomk::k_step<TPB, TEAMS>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc; }
    const unsigned grid = unsigned((P.n_envs + TPB - 1) / TPB);
    pomk::k_step<TPB, TEAMS><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, on ? on : b->stream>>>(P, reinterpret_cast<const uint32_t*>(moves_dev), flags, status_dev);
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

template<int TPB, bool TEAMS = false, bool FOG = false>
int launch_rollout(pom_batch* b, uint32_t ticks, uint64_t seed, uint32_t tick0, uint32_t flags, const uint8_t* move_seq = nullptr)
{
    const uint32_t n_actions = (flags & POM_ROLL_HARMLESS) ? 5u : 6u, no_reset = flags & (POM_ROLL_NO_RESET | POM_ROLL_CONTINUE_UNDEFINED);
    const uint32_t mask = (flags >> POM_ROLL_SIMPLE_SHIFT) & 0xFu;
    const unsigned grid = unsigned((b->n_envs + TPB - 1) / TPB);
    if(mask)
    {
        int rc = set_smem(b, attr_bit(ATTR_ROLLOUT_POLICY, TEAMS, FOG), pomk::k_rollout<TPB, true, false, TEAMS, FOG>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc;
        rc = ensure_policy(b); if(rc) return rc;
        pomk::k_rollout<TPB, true, false, TEAMS, FOG><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), ticks, seed, tick0, n_actions, no_reset,
                                                                                                     FOG ? mask | policy_view_bits(b) : mask, nullptr);
    }
    else if(!TEAMS && n_actions == 6u && no_reset == 0u && !move_seq && !b->no_spec)      /* the SPEC image is free-for-all only */
    {
        int rc = set_smem(b, ATTR_ROLLOUT_SPEC, pomk::k_rollout<TPB, false, true>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc;
        pomk::k_rollout<TPB, false, true><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), ticks, seed, tick0, 6u, 0u, 0u, nullptr);
    }
    else
    {
        int rc = set_smem(b, attr_bit(ATTR_ROLLOUT, TEAMS), pomk::k_rollout<TPB, false, false, TEAMS>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc;
        pomk::k_rollout<TPB, false, false, TEAMS><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), ticks, seed, tick0, n_actions, no_reset, 0u, reinterpret_cast<const uint32_t*>(move_seq));
    }
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

template<int TPB, bool TEAMS = false, bool FOG = false>
int launch_policy_moves(pom_batch* b, uint8_t* moves_dev, uint64_t seed, uint32_t tick, uint32_t mask, uint32_t gen_actions = 0, uint32_t freeze_truncated = 0)
{
    { int rc = set_smem(b, attr_bit(ATTR_POLICY_MOVES, TEAMS, FOG), pomk::k_policy_moves<TPB, TEAMS, FOG>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc; }
    const unsigned grid = unsigned((b->n_envs + TPB - 1) / TPB);
    pomk::k_policy_moves<TPB, TEAMS, FOG><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), reinterpret_cast<uint32_t*>(moves_dev), seed, tick,
                                                                                            FOG ? mask | policy_view_bits(b) : mask, gen_actions, freeze_truncated);
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

template<int TPB, bool RADIO = false>
int launch_observe_planes(pom_batch* b, uint8_t* obs_dev, uint32_t mask, int view, uint32_t cropped_bytes = 0)
{
    const unsigned grid = unsigned((b->n_envs + TPB - 1) / TPB);
    /* start where the last whole-batch step ended (its records are still in L2): a forward walk ended at the last tile */
    const uint32_t reverse = (b->pingpong && b->walk && ((b->walk - 1u) & 1u) == 0u) ? 1u : 0u;
    if(cropped_bytes)
    {
        int rc = set_smem(b, RADIO ? ATTR_OBS_CROPPED_RADIO : ATTR_OBS_CROPPED, pomk::k_observe_planes<TPB, true, RADIO>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc;
        pomk::k_observe_planes<TPB, true, RADIO><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), obs_dev, b->n_alloc, mask, view, reverse, cropped_bytes);
    }
    else
    {
        int rc = set_smem(b, RADIO ? ATTR_OBS_RADIO : ATTR_OBS, pomk::k_observe_planes<TPB, false, RADIO>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc;
        pomk::k_observe_planes<TPB, false, RADIO><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, b->stream>>>(b->params(), obs_dev, b->n_alloc, mask, view, reverse, 0u);
    }
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

template<int TPB, bool TEAMS = false>
int launch_expand(pom_batch* dst, const pom_batch* src, const uint32_t* idx_dev, uint64_t n_children, uint32_t fanout, uint32_t flags)
{
    { int rc = set_smem(dst, attr_bit(ATTR_EXPAND, TEAMS), pomk::k_expand_step<TPB, TEAMS>, pomk::TileScratch<TPB>::BYTES); if(rc) return rc; }
    const unsigned grid = unsigned((n_children + TPB - 1) / TPB);
    pomk::k_expand_step<TPB, TEAMS><<<grid, TPB, pomk::TileScratch<TPB>::BYTES, dst->stream>>>(dst->recs, src->recs, idx_dev, n_children, fanout, flags);
    dst->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

}

namespace
{
/* a caller's buffer as the device sees it: device memory as is, mapped pinned host memory through its device alias */
template<typename T>
int device_view(T* p, T** out, const char* what)
{
    *out = nullptr;
    if(!p) return POM_OK;
    cudaPointerAttributes a;
    if(cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return fail(POM_E_ARG, what); }
    if(a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) { *out = p; return POM_OK; }
    if(a.type == cudaMemoryTypeHost && a.devicePointer) { *out = static_cast<T*>(a.devicePointer); return POM_OK; }
    return fail(POM_E_ARG, what);
}
}

namespace
{
/* CPUs local to the GPU, from sysfs; empty when unknown */
bool local_cpus(int device, cpu_set_t* set)
{
    char bus[32] = {0};
    if(cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return false; }
    for(char* c = bus; *c; c++) if(*c >= 'A' && *c <= 'Z') *c = char(*c - 'A' + 'a');
    std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist");
    std::string list;
    if(!f || !std::getline(f, list) || list.empty()) return false;
    CPU_ZERO(set);
    int n = 0;
    size_t i = 0;
    while(i < list.size())
    {
        char* end = nullptr;
        const long lo = std::strtol(list.c_str() + i, &end, 10);
        long hi = lo;
        i = size_t(end - list.c_str());
        if(i < list.size() && list[i] == '-') { hi = std::strtol(list.c_str() + i + 1, &end, 10); i = size_t(end - list.c_str()); }
        for(long c = lo; c <= hi && c < CPU_SETSIZE; c++) { CPU_SET(int(c), set); n++; }
        if(i < list.size() && list[i] == ',') i++;
        else if(i < list.size() && (list[i] < '0' || list[i] > '9')) break;
    }
    return n > 0;
}
}

/* tile geometry: threads (= envs) per CTA; tunable through POM_TPB for experiments, default = measured best */
#define POM_DISPATCH(h, fn, ...) \
    do { \
        if((h)->tpb == 32) return fn<32>(__VA_ARGS__); \
        if((h)->tpb == 64) return fn<64>(__VA_ARGS__); \
        if((h)->tpb == 256) return fn<256>(__VA_ARGS__); \
        return fn<128>(__VA_ARGS__); \
    } while(0)
/* the same for the launches that step or act: a team handle takes the team images, which exist for the default
 * geometry only (POM_TPB does not apply to it) */
#define POM_DISPATCH_MODE(h, fn, ...) \
    do { \
        if((h)->teams) return fn<128, true>(__VA_ARGS__); \
        POM_DISPATCH(h, fn, __VA_ARGS__); \
    } while(0)
/* the same for the launches that run the device SimpleAgent: a handle with a policy view takes the FOG images of its mode,
 * which also exist for the default geometry only */
#define POM_DISPATCH_POLICY(h, fn, ...) \
    do { \
        if((h)->policy_view >= 0) \
        { \
            if((h)->teams) return fn<128, true, true>(__VA_ARGS__); \
            return fn<128, false, true>(__VA_ARGS__); \
        } \
        POM_DISPATCH_MODE(h, fn, __VA_ARGS__); \
    } while(0)

/* the observation planes of a handle: a radio handle takes the RADIO images, which exist for the default geometry only
 * (POM_TPB does not apply to it) */
static int launch_observe(pom_batch* b, uint8_t* obs_dev, uint32_t mask, int view, uint32_t cropped_bytes = 0)
{
    if(b->radio) return launch_observe_planes<128, true>(b, obs_dev, mask, view, cropped_bytes);
    POM_DISPATCH(b, launch_observe_planes, b, obs_dev, mask, view, cropped_bytes);
}

extern "C" {

const char* pom_last_error(void) { return g_err.c_str(); }

int pom_device_count(void)
{
    int n = 0;
    if(cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int pom_batch_init(pom_batch** out, int device, uint64_t n_envs, const pom_init_desc* desc)
{
    if(!out || !desc || n_envs == 0 || desc->n_templates == 0) return fail(POM_E_ARG, "pom_batch_init: bad argument");
    if(n_envs > (uint64_t(1) << 31)) return fail(POM_E_ARG, "pom_batch_init: too many envs for one handle");
    if((desc->flags & POM_INIT_RADIO) && !(desc->flags & POM_INIT_TEAMS))
        return fail(POM_E_ARG, "pom_batch_init: POM_INIT_RADIO needs POM_INIT_TEAMS (the radio talks to a teammate)");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if(ce != cudaSuccess || ndev == 0) return fail(POM_E_CUDA, "no CUDA device: the step path has no CPU fallback", ce);
    if(device < 0 || device >= ndev) return fail(POM_E_ARG, "pom_batch_init: no such device");
    CK(cudaSetDevice(device));
    pom_batch* b = new(std::nothrow) pom_batch();
    if(!b) return fail(POM_E_NOMEM, "host allocation failed");
    b->device = device;
    b->n_envs = n_envs;
    b->n_alloc = (n_envs + TILE_ALIGN - 1) / TILE_ALIGN * TILE_ALIGN;
    b->env_offset = desc->env_offset;
    b->n_templates = desc->n_templates;
    b->max_ticks = desc->max_ticks;
    b->teams = (desc->flags & POM_INIT_TEAMS) != 0;
    b->radio = (desc->flags & POM_INIT_RADIO) != 0;
    cudaDeviceGetAttribute(&b->n_sms, cudaDevAttrMultiProcessorCount, device);
    if(b->n_sms < 1) b->n_sms = 1;
    if(const char* e = std::getenv("POM_STEP_KERNEL")) b->step_kernel = std::strcmp(e, "tile") == 0 ? 1 : 0;
    if(const char* e = std::getenv("POM_WS_NW")) b->ws_nw = std::atoi(e);
    if(const char* e = std::getenv("POM_STEP_PINGPONG")) b->pingpong = std::atoi(e) != 0;
    if(const char* e = std::getenv("POM_OBS_FUSED")) b->obs_fused = std::atoi(e) != 0;
    if(const char* e = std::getenv("POM_WS_NOSPEC")) b->no_spec = std::atoi(e) != 0;
    if(const char* e = std::getenv("POM_ROLL_POLICY")) b->policy_pertick = std::strcmp(e, "fused") != 0;
    if(const char* e = std::getenv("POM_TPB"))
    {
        const int t = std::atoi(e);
        if(t == 32 || t == 64 || t == 128 || t == 256) b->tpb = t;
    }
    if(const char* e = std::getenv("POM_STEP_PARTS"))
    {
        const int p = std::atoi(e);
        if(p >= 2 && p <= 16) b->step_parts = p;
    }
    if(const char* e = std::getenv("POM_CHUNKS"))
    {
        const int c = std::atoi(e);
        if(c >= 1 && c <= pom_batch::MAX_CHUNKS) b->chunks = c;
    }
    if(const char* e = std::getenv("POM_ZEROCOPY")) b->zerocopy = std::atoi(e);
    int rc = POM_OK;
    do {
        if(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess ||
           cudaEventCreate(&b->ev[0]) != cudaSuccess || cudaEventCreate(&b->ev[1]) != cudaSuccess ||
           cudaStreamCreateWithFlags(&b->s_h2d, cudaStreamNonBlocking) != cudaSuccess ||
           cudaStreamCreateWithFlags(&b->s_d2h, cudaStreamNonBlocking) != cudaSuccess ||
           cudaStreamCreateWithFlags(&b->s_k2, cudaStreamNonBlocking) != cudaSuccess ||
           cudaEventCreateWithFlags(&b->ev_k2, cudaEventDisableTiming) != cudaSuccess ||
           cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming) != cudaSuccess ||
           cudaEventCreateWithFlags(&b->ev_begin, cudaEventDisableTiming) != cudaSuccess)
        { rc = fail(POM_E_CUDA, "stream/event creation failed", cudaGetLastError()); break; }
        if(alloc_records(device, b->n_alloc * POM_REC_BYTES, &b->recs, &b->recs_mapped) != cudaSuccess ||
           cudaMalloc(&b->templates, size_t(b->n_templates) * POM_REC_BYTES) != cudaSuccess ||
           cudaMalloc(&b->episodes, b->n_alloc * sizeof(uint32_t)) != cudaSuccess ||
           cudaMalloc(&b->stats, POM_STATS_WORDS * sizeof(unsigned long long)) != cudaSuccess ||
           cudaMalloc(&b->moves_buf, b->n_alloc * 4) != cudaSuccess ||
           cudaMalloc(&b->status_buf, b->n_alloc) != cudaSuccess)
        { rc = fail(POM_E_NOMEM, "device allocation failed", cudaGetLastError()); break; }
        if(cudaMemsetAsync(b->recs, 0, b->n_alloc * POM_REC_BYTES, b->stream) != cudaSuccess ||
           cudaMemsetAsync(b->episodes, 0, b->n_alloc * sizeof(uint32_t), b->stream) != cudaSuccess ||
           cudaMemsetAsync(b->stats, 0, POM_STATS_WORDS * sizeof(unsigned long long), b->stream) != cudaSuccess)
        { rc = fail(POM_E_CUDA, "memset failed", cudaGetLastError()); break; }
        if(desc->host_templates)
        {
            uint32_t bad = 0;
            rc = pack_into(b, b->templates, 0, b->n_templates, desc->host_templates, nullptr, &bad);
            if(rc) break;
            if(bad) { rc = fail(POM_E_STATE, "a host template cannot be represented in the packed record"); break; }
        }
        else
        {
            rc = build_templates_from_seeds(b, desc->first_seed);
            if(rc) break;
        }
        if(!(desc->flags & POM_INIT_EMPTY))
        {
            rc = fill_from_templates(b);
            if(rc) break;
        }
        if(cudaStreamSynchronize(b->stream) != cudaSuccess) { rc = fail(POM_E_CUDA, "init sync failed", cudaGetLastError()); break; }
    } while(0);
    if(rc) { pom_batch_destroy(b); return rc; }
    *out = b;
    return POM_OK;
}

int pom_batch_destroy(pom_batch* b)
{
    if(!b) return POM_OK;
    cudaSetDevice(b->device);
    if(b->s_k2) cudaStreamSynchronize(b->s_k2);
    if(b->stream) cudaStreamSynchronize(b->stream);
    free_records(b->recs, b->recs_mapped); cudaFree(b->templates); cudaFree(b->episodes); cudaFree(b->stats);
    cudaFree(b->moves_buf); cudaFree(b->status_buf); cudaFree(b->aos_stage); cudaFree(b->st_stage);
    cudaFree(b->bad_count); cudaFree(b->flush_buf); cudaFree(b->idx_buf); if(b->ev_expand) cudaEventDestroy(b->ev_expand); cudaFree(b->policy); cudaFree(b->fin_counter);
    if(b->ev[0]) cudaEventDestroy(b->ev[0]);
    if(b->ev[1]) cudaEventDestroy(b->ev[1]);
    for(int i = 0; i < pom_batch::MAX_CHUNKS; i++) { if(b->ev_in[i]) cudaEventDestroy(b->ev_in[i]); if(b->ev_done[i]) cudaEventDestroy(b->ev_done[i]); }
    if(b->ev_out) cudaEventDestroy(b->ev_out);
    if(b->ev_begin) cudaEventDestroy(b->ev_begin);
    if(b->s_h2d) cudaStreamDestroy(b->s_h2d);
    if(b->s_d2h) cudaStreamDestroy(b->s_d2h);
    if(b->s_k2) cudaStreamDestroy(b->s_k2);
    if(b->ev_k2) cudaEventDestroy(b->ev_k2);
    if(b->stream) cudaStreamDestroy(b->stream);
    delete b;
    return POM_OK;
}

int pom_batch_sync(pom_batch* b)
{
    int rc = use(b); if(rc) return rc;
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_upload(pom_batch* b, uint64_t first, uint64_t count, const pom_state* states, const uint8_t* status)
{
    int rc = use(b); if(rc) return rc;
    if(!states) return fail(POM_E_ARG, "pom_batch_upload: null states");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_upload: range outside the batch");
    uint32_t bad = 0;
    rc = pack_into(b, b->recs, first, count, states, status, &bad);
    if(rc) return rc;
    if(bad) return fail(POM_E_STATE, "pom_batch_upload: some states cannot be represented (marked POM_STATUS_INVALID)");
    return POM_OK;
}

int pom_batch_download(pom_batch* b, uint64_t first, uint64_t count, pom_state* states, uint8_t* status)
{
    int rc = use(b); if(rc) return rc;
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_download: range outside the batch");
    rc = ensure_stage(b); if(rc) return rc;
    for(uint64_t done = 0; done < count; done += XFER_CHUNK)
    {
        const uint64_t c = count - done < XFER_CHUNK ? count - done : XFER_CHUNK;
        pomk::k_unpack<<<unsigned((c + 127) / 128), 128, 0, b->stream>>>(b->recs, states ? b->aos_stage : nullptr, b->st_stage, first + done, c);
        b->launches++;
        CK(cudaGetLastError());
        if(states) CK(cudaMemcpyAsync(states + done, b->aos_stage, c * sizeof(pom_state), cudaMemcpyDeviceToHost, b->stream));
        if(status) CK(cudaMemcpyAsync(status + done, b->st_stage, c, cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
    }
    return POM_OK;
}

int pom_batch_observe(pom_batch* b, uint64_t first, uint64_t count, int agent, int view, pom_state* states, uint8_t* status)
{
    int rc = use(b); if(rc) return rc;
    if(!states) return fail(POM_E_ARG, "pom_batch_observe: null output");
    if(agent < 0 || agent > 3 || view < 0) return fail(POM_E_ARG, "pom_batch_observe: agent must be 0..3 and view >= 0");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_observe: range outside the batch");
    rc = ensure_stage(b); if(rc) return rc;
    for(uint64_t done = 0; done < count; done += XFER_CHUNK)
    {
        const uint64_t c = count - done < XFER_CHUNK ? count - done : XFER_CHUNK;
        pomk::k_observe<<<unsigned((c + 127) / 128), 128, 0, b->stream>>>(b->recs, b->aos_stage, b->st_stage, first + done, c, agent, view);
        b->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(states + done, b->aos_stage, c * sizeof(pom_state), cudaMemcpyDeviceToHost, b->stream));
        if(status) CK(cudaMemcpyAsync(status + done, b->st_stage, c, cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
    }
    return POM_OK;
}

uint64_t pom_batch_obs_stride(const pom_batch* b) { return b ? b->n_alloc : 0; }

int pom_batch_observe_planes(pom_batch* b, uint8_t* obs_dev, uint32_t agent_mask, int view)
{
    int rc = use(b); if(rc) return rc;
    if(!obs_dev) return fail(POM_E_ARG, "pom_batch_observe_planes: null output");
    if(agent_mask == 0 || agent_mask > 0xFu || view < 0) return fail(POM_E_ARG, "pom_batch_observe_planes: agent_mask must be 1..15 and view >= 0");
    return launch_observe(b, obs_dev, agent_mask, view);
}

int pom_device_copy(int device, void* dst, const void* src, uint64_t bytes)
{
    if(!dst || !src) return fail(POM_E_ARG, "pom_device_copy: null pointer");
    CK(cudaSetDevice(device));
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDefault));
    return POM_OK;
}

int pom_batch_reset(pom_batch* b)
{
    int rc = use(b); if(rc) return rc;
    CK(cudaMemsetAsync(b->episodes, 0, b->n_alloc * sizeof(uint32_t), b->stream));
    CK(cudaMemsetAsync(b->stats, 0, POM_STATS_WORDS * sizeof(unsigned long long), b->stream));
    if(b->policy) CK(cudaMemsetAsync(b->policy, 0, 9 * b->n_alloc * sizeof(uint32_t), b->stream));
    return fill_from_templates(b);
}

int pom_batch_templates(pom_batch* b, pom_state* out, int32_t* seeds_out)
{
    int rc = use(b); if(rc) return rc;
    if(!out) return fail(POM_E_ARG, "pom_batch_templates: null output");
    rc = ensure_stage(b); if(rc) return rc;
    for(uint64_t done = 0; done < b->n_templates; done += XFER_CHUNK)
    {
        const uint64_t c = b->n_templates - done < XFER_CHUNK ? b->n_templates - done : XFER_CHUNK;
        pomk::k_unpack<<<unsigned((c + 127) / 128), 128, 0, b->stream>>>(b->templates, b->aos_stage, b->st_stage, done, c);
        b->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out + done, b->aos_stage, c * sizeof(pom_state), cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));
    }
    if(seeds_out)
    {
        for(uint32_t k = 0; k < b->n_templates; k++) seeds_out[k] = k < b->seeds.size() ? b->seeds[k] : 0;
    }
    return POM_OK;
}

int pom_batch_step(pom_batch* b, const uint8_t* moves_dev, uint32_t flags)
{
    const bool overlap = (flags & POM_STEP_OVERLAP) && b && b->n_envs >= (uint64_t(1) << 18);
    int rc = use(b, !overlap); if(rc) return rc;
    if(!moves_dev) return fail(POM_E_ARG, "pom_batch_step: null moves");
    if(!overlap) POM_DISPATCH_MODE(b, launch_step, b, moves_dev, flags, nullptr);
    /* Two halves on two streams.  The second half waits for everything queued on the handle's stream so far (the
     * caller's moves, the first half of the previous tick) and, by stream order, for its own previous tick; the first
     * half of the NEXT tick does not wait for it.  So the last, partly filled wave of one kernel runs next to the first
     * wave of the other, tick after tick; use() joins the streams before any other operation. */
    const int parts = b->step_parts;
    const uint64_t per = ((b->n_envs + parts - 1) / parts + 1023) / 1024 * 1024;
    /* Up to 0.5 Mi envs the two parts run on the tile kernel: its small CTAs let the two launches share every SM (the
     * persistent kernel takes a whole SM per CTA, so its two launches can only follow each other), and with 60 slices or
     * fewer per SM the persistent launch is mostly fill and drain: 0.047 against 0.057 ms per tick at 0.5 Mi envs, 0.031
     * against 0.034 at 0.25 Mi (tools/prof_step.py).  Same tick code, same results. */
    const bool tile_parts = b->n_envs <= (uint64_t(1) << 19) && !b->no_spec;
    CK(cudaEventRecord(b->ev_begin, b->stream));
    CK(cudaStreamWaitEvent(b->s_k2, b->ev_begin, 0));
    int c = 0;
    for(uint64_t first = 0; first < b->n_envs; first += per, c++)
    {
        const uint64_t count = first + per <= b->n_envs ? per : b->n_envs - first;
        rc = [&]() -> int { POM_DISPATCH_MODE(b, launch_step, b, moves_dev, flags, nullptr, first, count, (c & 1) ? b->s_k2 : b->stream, tile_parts); }();
        if(rc) return rc;
    }
    b->forked = true;
    return POM_OK;
}

/* The chunked pipeline of pom_batch_step_host over four streams: copy-in, two compute streams (chunks alternate, so
 * that the partial last wave of one chunk's kernel overlaps the first wave of the next), copy-out.
 * The kernel itself writes the end-of-tick status bytes (before any auto-reset), so no extra pass is needed for them.
 * Ends with every forked stream joined back into the handle's stream. */
static int enqueue_step_pipeline(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags, int chunks, uint64_t per)
{
    const uint64_t n = b->n_envs;
    /* everything already queued on the handle's stream happens before this step */
    CK(cudaEventRecord(b->ev_begin, b->stream));
    CK(cudaStreamWaitEvent(b->s_h2d, b->ev_begin, 0));
    if(chunks > 1) CK(cudaStreamWaitEvent(b->s_k2, b->ev_begin, 0));
    for(int c = 0; c < chunks; c++)
    {
        const uint64_t first = uint64_t(c) * per, count = (first + per <= n) ? per : n - first;
        cudaStream_t compute = (c & 1) ? b->s_k2 : b->stream;     /* chunks are independent (disjoint envs) */
        CK(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(b->moves_buf) + 4 * first, moves_host + 4 * first, 4 * count, cudaMemcpyHostToDevice, b->s_h2d));
        CK(cudaEventRecord(b->ev_in[c], b->s_h2d));
        CK(cudaStreamWaitEvent(compute, b->ev_in[c], 0));
        const int rc = [&]() -> int { POM_DISPATCH_MODE(b, launch_step, b, reinterpret_cast<const uint8_t*>(b->moves_buf), flags,
                                                   status_host ? b->status_buf : nullptr, first, count, compute); }();
        if(rc) return rc;
        if(status_host)
        {
            CK(cudaEventRecord(b->ev_done[c], compute));
            CK(cudaStreamWaitEvent(b->s_d2h, b->ev_done[c], 0));
            CK(cudaMemcpyAsync(status_host + first, b->status_buf + first, count, cudaMemcpyDeviceToHost, b->s_d2h));
        }
    }
    if(chunks > 1)
    {
        CK(cudaEventRecord(b->ev_k2, b->s_k2));
        CK(cudaStreamWaitEvent(b->stream, b->ev_k2, 0));
    }
    if(status_host)
    {
        CK(cudaEventRecord(b->ev_out, b->s_d2h));
        CK(cudaStreamWaitEvent(b->stream, b->ev_out, 0));
    }
    return POM_OK;
}

/* zero-copy launch shared by pom_batch_step_host (pinned buffers) and pom_batch_step_host_async; returns 1 if the buffers
 * are not page-locked/mapped (nothing launched), 0 on success, a negative POM_E_* on error */
static int launch_step_zero_copy(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags)
{
    void* mdev = nullptr; void* sdev = nullptr;
    bool ok = cudaHostGetDevicePointer(&mdev, const_cast<uint8_t*>(moves_host), 0) == cudaSuccess;
    if(ok && status_host) ok = cudaHostGetDevicePointer(&sdev, status_host, 0) == cudaSuccess;
    if(!ok) { cudaGetLastError(); return 1; }
    return [&]() -> int { POM_DISPATCH_MODE(b, launch_step, b, static_cast<const uint8_t*>(mdev), flags, static_cast<uint8_t*>(sdev)); }();
}

int pom_batch_step_host_async(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_host) return fail(POM_E_ARG, "pom_batch_step_host_async: null moves");
    rc = launch_step_zero_copy(b, moves_host, status_host, flags);
    if(rc == 1) return fail(POM_E_ARG, "pom_batch_step_host_async: the buffers must be page-locked, device-mapped memory (pom_host_alloc)");
    return rc;
}

int pom_batch_step_host(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_host) return fail(POM_E_ARG, "pom_batch_step_host: null moves");
    const uint64_t n = b->n_envs;
    /* Pinned (page-locked, mapped) host buffers: the kernel reads the move bytes from and writes the status bytes to host
     * memory itself (its one coalesced load per warp is issued before the wait for the bulk state copy, so the PCIe
     * latency hides behind it); no staging copies, no chunks.  POM_ZEROCOPY=0 forces the copy pipeline. */
    if(b->zerocopy)
    {
        rc = launch_step_zero_copy(b, moves_host, status_host, flags);
        if(rc < 0) return rc;
        if(rc == 0)
        {
            CK(cudaStreamSynchronize(b->stream));
            return POM_OK;
        }
        /* pageable memory: fall through to the copy pipeline */
    }
    /* Pageable buffers: staged copies.  POM_CHUNKS is a tuning knob for experiments; the default is the measured best for 1 Mi envs (6 chunks on two
     * compute streams: 175 us per tick against 219 us for 3 chunks on one stream; submitting the same pipeline as a
     * CUDA graph was measured too and is slower than the direct calls, 182 us) */
    int chunks = n >= (uint64_t(1) << 18) ? b->chunks : 1;
    const uint64_t per = ((n + chunks - 1) / chunks + 1023) / 1024 * 1024;      /* multiple of every TPB */
    chunks = int((n + per - 1) / per);
    for(int c = 0; c < chunks; c++)
    {
        if(!b->ev_in[c])
        {
            CK(cudaEventCreateWithFlags(&b->ev_in[c], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&b->ev_done[c], cudaEventDisableTiming));
        }
    }
    rc = enqueue_step_pipeline(b, moves_host, status_host, flags, chunks, per);
    if(rc) return rc;
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

uint32_t pom_obs_cropped_bytes(int view) { return (view < 0 || view > 5) ? 0u : pomcore::obs_cropped_bytes(view); }

int pom_batch_observe_planes_cropped(pom_batch* b, uint8_t* obs_dev, uint32_t agent_mask, int view)
{
    int rc = use(b); if(rc) return rc;
    if(!obs_dev) return fail(POM_E_ARG, "pom_batch_observe_planes_cropped: null output");
    if(agent_mask == 0 || agent_mask > 0xFu || view < 0 || view > 5) return fail(POM_E_ARG, "pom_batch_observe_planes_cropped: agent_mask must be 1..15 and view 0..5");
    return launch_observe(b, obs_dev, agent_mask, view, pomcore::obs_cropped_bytes(view));
}

int pom_batch_step_observe(pom_batch* b, const uint8_t* moves_dev, uint32_t flags, uint8_t* obs_dev, uint32_t agent_mask, int view)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_dev || !obs_dev) return fail(POM_E_ARG, "pom_batch_step_observe: null pointer");
    if(agent_mask == 0 || agent_mask > 0xFu || view < 0) return fail(POM_E_ARG, "pom_batch_step_observe: agent_mask must be 1..15 and view >= 0");
    if(flags & POM_STEP_OVERLAP) return fail(POM_E_ARG, "pom_batch_step_observe: POM_STEP_OVERLAP is not supported");
    if(b->step_kernel != 0) return fail(POM_E_ARG, "pom_batch_step_observe needs the persistent step kernel (unset POM_STEP_KERNEL)");
    pomk::StepIO k{};
    k.moves = moves_dev;
    /* the fused images have no radio: a radio handle always takes the two launches */
    if(b->obs_fused && !b->radio)
    {
        k.obs = obs_dev; k.obs_stride = b->n_alloc; k.obs_mask = agent_mask; k.obs_view = view;
        return launch_step_io(b, b->params(), k, flags, b->stream);
    }
    /* Two launches, the second one starting with the records the first one wrote last.  Writing the planes from inside
     * the step kernel saves the second read of the records, but the slice buffers are then held for twice as long and 24
     * of them per SM no longer cover the latency: 0.267 ms per 1 Mi envs against 0.104 + 0.135 ms (DESIGN section 8). */
    rc = launch_step_io(b, b->params(), k, flags, b->stream);
    if(rc) return rc;
    return launch_observe(b, obs_dev, agent_mask, view);
}

int pom_batch_step_compact(pom_batch* b, const pom_step_compact_io* io, uint32_t flags)
{
    int rc = use(b); if(rc) return rc;
    if(!io || !io->joint) return fail(POM_E_ARG, "pom_batch_step_compact: null joint actions");
    if(io->fin_env && (!io->fin_status || !io->fin_count)) return fail(POM_E_ARG, "pom_batch_step_compact: fin_env needs fin_status and fin_count");
    if(flags & POM_STEP_OVERLAP) return fail(POM_E_ARG, "pom_batch_step_compact: POM_STEP_OVERLAP is not supported");
    if(b->step_kernel != 0) return fail(POM_E_ARG, "pom_batch_step_compact needs the persistent step kernel (unset POM_STEP_KERNEL)");
    pomk::StepIO k{};
    uint16_t* joint = nullptr; uint32_t* count = nullptr;
    const char* bad = "pom_batch_step_compact: buffers must be device memory or page-locked mapped host memory (pom_host_alloc)";
    if((rc = device_view(const_cast<uint16_t*>(io->joint), &joint, bad))) return rc;
    if((rc = device_view(io->done_bits, &k.done_bits, bad))) return rc;
    if((rc = device_view(io->fin_env, &k.fin_env, bad))) return rc;
    if((rc = device_view(io->fin_status, &k.fin_status, bad))) return rc;
    if((rc = device_view(io->fin_count, &count, bad))) return rc;
    k.moves = joint;
    k.joint = 1u;
    k.fin_capacity = io->fin_capacity;
    if(io->obs_dev)
    {
        if(io->obs_agent_mask == 0 || io->obs_agent_mask > 0xFu || io->obs_view < 0) return fail(POM_E_ARG, "pom_batch_step_compact: obs_agent_mask must be 1..15 and obs_view >= 0");
        if(b->obs_fused && !b->radio) { k.obs = io->obs_dev; k.obs_stride = b->n_alloc; k.obs_mask = io->obs_agent_mask; k.obs_view = io->obs_view; }
    }
    if(k.fin_env)
    {
        if(!b->fin_counter)
        {
            CK(cudaMalloc(&b->fin_counter, 2 * sizeof(uint32_t)));
            CK(cudaMemsetAsync(b->fin_counter, 0, 2 * sizeof(uint32_t), b->stream));
        }
        k.fin_counter = b->fin_counter;
        k.fin_count_out = count;
    }
    rc = launch_step_io(b, b->params(), k, flags, b->stream);
    if(rc || !io->obs_dev || k.obs) return rc;
    return launch_observe(b, io->obs_dev, io->obs_agent_mask, io->obs_view);
}

int pom_batch_step_rewards(pom_batch* b, const uint8_t* moves_dev, uint32_t flags, int8_t* rewards, uint8_t* status)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_dev || !rewards) return fail(POM_E_ARG, "pom_batch_step_rewards: null moves or rewards");
    if(flags & ~uint32_t(POM_STEP_AUTORESET | POM_STEP_COUNT | POM_STEP_CONTINUE_UNDEFINED))
        return fail(POM_E_ARG, "pom_batch_step_rewards: only POM_STEP_AUTORESET, POM_STEP_COUNT and POM_STEP_CONTINUE_UNDEFINED are accepted");
    if(b->step_kernel != 0) return fail(POM_E_ARG, "pom_batch_step_rewards needs the persistent step kernel (unset POM_STEP_KERNEL)");
    pomk::StepIO k{};
    uint8_t* moves = nullptr; int8_t* rw = nullptr;
    const char* bad = "pom_batch_step_rewards: buffers must be device memory or page-locked mapped host memory (pom_host_alloc)";
    if((rc = device_view(const_cast<uint8_t*>(moves_dev), &moves, bad))) return rc;
    if((rc = device_view(rewards, &rw, bad))) return rc;
    if((rc = device_view(status, &k.status_out, bad))) return rc;
    /* each env's four rewards are stored as one word */
    if(reinterpret_cast<uintptr_t>(rw) & 3u) return fail(POM_E_ARG, "pom_batch_step_rewards: rewards must be 4-byte aligned");
    k.moves = moves;
    k.obs = reinterpret_cast<uint8_t*>(rw);                           /* the REWARDS images' output slot (StepIO::obs) */
    return launch_step_io(b, b->params(), k, flags, b->stream, true);
}

int pom_batch_step_radio(pom_batch* b, const uint8_t* moves_dev, const uint8_t* msgs, uint32_t flags, int8_t* rewards, uint8_t* status)
{
    int rc = use(b); if(rc) return rc;
    if(!b->radio) return fail(POM_E_ARG, "pom_batch_step_radio needs a handle made with POM_INIT_RADIO");
    if(!moves_dev || !msgs) return fail(POM_E_ARG, "pom_batch_step_radio: null moves or messages");
    if(flags & ~uint32_t(POM_STEP_AUTORESET | POM_STEP_COUNT | POM_STEP_CONTINUE_UNDEFINED))
        return fail(POM_E_ARG, "pom_batch_step_radio: only POM_STEP_AUTORESET, POM_STEP_COUNT and POM_STEP_CONTINUE_UNDEFINED are accepted");
    if(b->step_kernel != 0) return fail(POM_E_ARG, "pom_batch_step_radio needs the persistent step kernel (unset POM_STEP_KERNEL)");
    pomk::StepIO k{};
    uint8_t* moves = nullptr; uint8_t* m = nullptr; int8_t* rw = nullptr;
    const char* bad = "pom_batch_step_radio: buffers must be device memory or page-locked mapped host memory (pom_host_alloc)";
    if((rc = device_view(const_cast<uint8_t*>(moves_dev), &moves, bad))) return rc;
    if((rc = device_view(const_cast<uint8_t*>(msgs), &m, bad))) return rc;
    if((rc = device_view(rewards, &rw, bad))) return rc;
    if((rc = device_view(status, &k.status_out, bad))) return rc;
    /* each env's four message bytes are loaded, and its four rewards stored, as one word */
    if((reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(rw)) & 3u)
        return fail(POM_E_ARG, "pom_batch_step_radio: msgs and rewards must be 4-byte aligned");
    k.moves = moves;
    k.obs = reinterpret_cast<uint8_t*>(rw);                           /* the RADIO image's rewards slot (StepIO::obs), may be null */
    k.fin_status = m;                                                 /* its messages slot (StepIO::fin_status) */
    return launch_step_io(b, b->params(), k, flags, b->stream, true, true);
}

int pom_batch_rollout(pom_batch* b, uint32_t ticks, uint64_t rng_seed, uint32_t tick0, uint32_t flags)
{
    int rc = use(b); if(rc) return rc;
    const uint32_t mask = (flags >> POM_ROLL_SIMPLE_SHIFT) & 0xFu;
    if(mask && !(flags & POM_ROLL_NO_RESET) && b->policy_pertick && b->step_kernel == 0 && b->n_envs >= (uint64_t(1) << 16))
    {
        /* A large batch with SimpleAgents runs tick by tick: k_policy_moves (which also draws the other agents' random
         * moves) and the per-tick step kernel, two launches per tick on the records in HBM - the same moves, states and
         * counters as the fused kernel, 1.26 against 0.94 x 10^9 env-steps/s with four SimpleAgents on 1 Mi envs.  The
         * fused image (policy + tick, 7200 instructions, warps spread over both halves of it) is the slower one whatever
         * its register budget; policy work dwarfs the HBM traffic of a tick here. */
        rc = ensure_policy(b); if(rc) return rc;
        const uint32_t n_actions = (flags & POM_ROLL_HARMLESS) ? 5u : 6u;
        const uint32_t sflags = POM_STEP_AUTORESET | POM_STEP_COUNT | pomk::STEP_FREEZE_TRUNCATED |
                                ((flags & POM_ROLL_CONTINUE_UNDEFINED) ? uint32_t(POM_STEP_CONTINUE_UNDEFINED) : 0u);
        uint8_t* mv = reinterpret_cast<uint8_t*>(b->moves_buf);
        for(uint32_t k = 0; k < ticks; k++)
        {
            rc = [&]() -> int { POM_DISPATCH_POLICY(b, launch_policy_moves, b, mv, rng_seed, tick0 + k, mask, n_actions, 1u); }();
            if(rc) return rc;
            rc = [&]() -> int { POM_DISPATCH_MODE(b, launch_step, b, mv, sflags, nullptr); }();
            if(rc) return rc;
        }
        return POM_OK;
    }
    if(mask) POM_DISPATCH_POLICY(b, launch_rollout, b, ticks, rng_seed, tick0, flags);
    POM_DISPATCH_MODE(b, launch_rollout, b, ticks, rng_seed, tick0, flags);
}

int pom_batch_step_seq(pom_batch* b, const uint8_t* moves_dev, uint32_t ticks, uint32_t flags)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_dev) return fail(POM_E_ARG, "pom_batch_step_seq: null moves");
    if(flags & ~uint32_t(POM_ROLL_NO_RESET | POM_ROLL_CONTINUE_UNDEFINED)) return fail(POM_E_ARG, "pom_batch_step_seq: only POM_ROLL_NO_RESET and POM_ROLL_CONTINUE_UNDEFINED are accepted");
    POM_DISPATCH_MODE(b, launch_rollout, b, ticks, 0, 0, flags, moves_dev);
}

int pom_batch_policy_moves(pom_batch* b, uint8_t* moves_dev, uint64_t seed, uint32_t tick, uint32_t agent_mask)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_dev) return fail(POM_E_ARG, "pom_batch_policy_moves: null moves");
    if(agent_mask == 0 || agent_mask > 0xFu) return fail(POM_E_ARG, "pom_batch_policy_moves: agent_mask must be 1..15");
    rc = ensure_policy(b); if(rc) return rc;
    POM_DISPATCH_POLICY(b, launch_policy_moves, b, moves_dev, seed, tick, agent_mask);
}

int pom_batch_policy_moves_host(pom_batch* b, uint8_t* moves_host, uint64_t seed, uint32_t tick, uint32_t agent_mask)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_host) return fail(POM_E_ARG, "pom_batch_policy_moves_host: null moves");
    CK(cudaMemcpyAsync(b->moves_buf, moves_host, 4 * b->n_envs, cudaMemcpyHostToDevice, b->stream));
    rc = pom_batch_policy_moves(b, reinterpret_cast<uint8_t*>(b->moves_buf), seed, tick, agent_mask);
    if(rc) return rc;
    CK(cudaMemcpyAsync(moves_host, b->moves_buf, 4 * b->n_envs, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_policy_act(pom_batch* b, uint64_t env, int agent, int draw, int* move_out)
{
    int rc = use(b); if(rc) return rc;
    if(!move_out) return fail(POM_E_ARG, "pom_batch_policy_act: null output");
    if(env >= b->n_envs) return fail(POM_E_RANGE, "pom_batch_policy_act: env outside the batch");
    if(agent < 0 || agent > 3 || draw < 0 || draw > 4) return fail(POM_E_ARG, "pom_batch_policy_act: agent must be 0..3 and draw 0..4");
    rc = ensure_policy(b); if(rc) return rc;
    DevBuf dev;
    CK(dev.alloc(sizeof(int)));
    if(b->policy_view >= 0)
    {
        const uint32_t arg = uint32_t(draw) | policy_view_bits(b);
        if(b->teams) pomk::k_policy_act<true, true><<<1, 1, 0, b->stream>>>(b->params(), env, agent, arg, dev.as<int>());
        else pomk::k_policy_act<false, true><<<1, 1, 0, b->stream>>>(b->params(), env, agent, arg, dev.as<int>());
    }
    else if(b->teams) pomk::k_policy_act<true><<<1, 1, 0, b->stream>>>(b->params(), env, agent, uint32_t(draw), dev.as<int>());
    else pomk::k_policy_act<<<1, 1, 0, b->stream>>>(b->params(), env, agent, uint32_t(draw), dev.as<int>());
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(move_out, dev.p, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_policy_reset(pom_batch* b)
{
    int rc = use(b); if(rc) return rc;
    if(b->policy) CK(cudaMemsetAsync(b->policy, 0, 8 * b->n_alloc * sizeof(uint32_t), b->stream));
    /* word 8 (the episode tag) is left alone: zeroed memories are valid for any episode */
    return POM_OK;
}

int pom_batch_policy_download(pom_batch* b, uint64_t first, uint64_t count, pom_simple_agent* out)
{
    int rc = use(b); if(rc) return rc;
    if(!out) return fail(POM_E_ARG, "pom_batch_policy_download: null output");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_policy_download: range outside the batch");
    if(count == 0) return POM_OK;
    rc = ensure_policy(b); if(rc) return rc;
    DevBuf tmp;
    CK(tmp.alloc(count * 32));
    pomk::k_policy_export<<<unsigned((count + 127) / 128), 128, 0, b->stream>>>(b->params(), first, count, tmp.as<uint32_t>());
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, tmp.p, count * 32, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_policy_upload(pom_batch* b, uint64_t first, uint64_t count, const pom_simple_agent* in)
{
    int rc = use(b); if(rc) return rc;
    if(!in) return fail(POM_E_ARG, "pom_batch_policy_upload: null input");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_policy_upload: range outside the batch");
    if(count == 0) return POM_OK;
    rc = ensure_policy(b); if(rc) return rc;
    DevBuf tmp;
    CK(tmp.alloc(count * 32));
    CK(cudaMemcpyAsync(tmp.p, in, count * 32, cudaMemcpyHostToDevice, b->stream));
    pomk::k_policy_import<<<unsigned((count + 127) / 128), 128, 0, b->stream>>>(b->params(), first, count, tmp.as<uint32_t>());
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_clone(pom_batch* dst, uint64_t first_dst, const pom_batch* src, const uint32_t* src_idx, uint64_t n_dst)
{
    int rc = use(dst); if(rc) return rc;
    if(!src || !src_idx) return fail(POM_E_ARG, "pom_batch_clone: null argument");
    if(src->device != dst->device) return fail(POM_E_ARG, "pom_batch_clone: handles live on different devices");
    if(src->teams != dst->teams) return fail(POM_E_ARG, "pom_batch_clone: one handle plays the team game and the other free-for-all (status bytes mean different things)");
    if(src->radio != dst->radio) return fail(POM_E_ARG, "pom_batch_clone: one handle has the radio and the other not (a record's radio bytes would leak)");
    if(src != dst) { rc = use(src); if(rc) return rc; }         /* joins src's second compute stream if a step is in flight there */
    if(first_dst > dst->n_envs || n_dst > dst->n_envs - first_dst) return fail(POM_E_RANGE, "pom_batch_clone: destination range outside the batch");
    for(uint64_t i = 0; i < n_dst; i++) if(src_idx[i] >= src->n_envs) return fail(POM_E_RANGE, "pom_batch_clone: source index outside the batch");
    if(n_dst == 0) return POM_OK;
    DevBuf idx_b, snap;
    CK(idx_b.alloc(n_dst * sizeof(uint32_t)));
    uint32_t* idx_dev = idx_b.as<uint32_t>();
    CK(cudaMemcpyAsync(idx_dev, src_idx, n_dst * sizeof(uint32_t), cudaMemcpyHostToDevice, dst->stream));
    if(src != dst) CK(cudaStreamSynchronize(src->stream));
    const uint8_t* from = src->recs;
    if(src == dst)
    {
        /* in-place gather: read from a snapshot so overlapping ranges are well defined */
        CK(snap.alloc(dst->n_alloc * POM_REC_BYTES));
        CK(cudaMemcpyAsync(snap.p, dst->recs, dst->n_alloc * POM_REC_BYTES, cudaMemcpyDeviceToDevice, dst->stream));
        from = snap.as<uint8_t>();
    }
    const uint64_t words = n_dst * POM_REC_WORDS;
    pomk::k_gather_records<<<unsigned((words + 255) / 256), 256, 0, dst->stream>>>(
        reinterpret_cast<uint32_t*>(dst->recs), reinterpret_cast<const uint32_t*>(from), idx_dev, n_dst, first_dst);
    dst->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(dst->stream));
    return POM_OK;
}

int pom_batch_expand_step(pom_batch* dst, const pom_batch* src, const uint32_t* src_idx, uint64_t n_roots, uint32_t fanout, uint32_t flags)
{
    int rc = use(dst); if(rc) return rc;
    if(!src || !src_idx || src == dst) return fail(POM_E_ARG, "pom_batch_expand_step: bad argument");
    if(src->device != dst->device) return fail(POM_E_ARG, "pom_batch_expand_step: handles live on different devices");
    if(src->teams != dst->teams) return fail(POM_E_ARG, "pom_batch_expand_step: one handle plays the team game and the other free-for-all (status bytes mean different things)");
    if(src->radio != dst->radio) return fail(POM_E_ARG, "pom_batch_expand_step: one handle has the radio and the other not (a record's radio bytes would leak)");
    rc = use(src); if(rc) return rc;                              /* joins src's second compute stream if a step is in flight there */
    if(fanout == 0 || fanout > 1296) return fail(POM_E_ARG, "pom_batch_expand_step: fanout must be 1..1296");
    const uint64_t n_children = n_roots * fanout;
    if(n_children > dst->n_envs) return fail(POM_E_RANGE, "pom_batch_expand_step: destination too small");
    for(uint64_t i = 0; i < n_roots; i++) if(src_idx[i] >= src->n_envs) return fail(POM_E_RANGE, "pom_batch_expand_step: root index outside the batch");
    if(n_roots == 0) return POM_OK;
    /* the index array lives in a buffer of the handle that only grows: a cudaMalloc / cudaFree pair per call cost more
     * than the kernel of a small expansion, and the call no longer has to wait for the kernel before returning */
    if(dst->idx_cap < n_roots)
    {
        CK(cudaStreamSynchronize(dst->stream));
        if(dst->idx_buf) CK(cudaFree(dst->idx_buf));
        dst->idx_buf = nullptr; dst->idx_cap = 0;
        if(cudaMalloc(reinterpret_cast<void**>(&dst->idx_buf), n_roots * sizeof(uint32_t)) != cudaSuccess)
            return fail(POM_E_NOMEM, "pom_batch_expand_step: index buffer");
        dst->idx_cap = n_roots;
    }
    uint32_t* idx_dev = dst->idx_buf;
    /* pageable source: the runtime has read src_idx when this returns; the copy itself is ordered on dst's stream,
     * behind the kernel of a previous expansion that may still be reading the buffer */
    CK(cudaMemcpyAsync(idx_dev, src_idx, n_roots * sizeof(uint32_t), cudaMemcpyHostToDevice, dst->stream));
    CK(cudaStreamSynchronize(src->stream));
    /* the mode is the source's (the kernel takes no BatchParams); the two handles' modes are equal */
    rc = [&]() -> int {
        if(src->teams) return launch_expand<128, true>(dst, src, idx_dev, n_children, fanout, flags);
        POM_DISPATCH(dst, launch_expand, dst, src, idx_dev, n_children, fanout, flags);
    }();
    if(rc) return rc;
    /* the call returns with the kernel queued: whatever is queued on the SOURCE handle from now on (a step that rewrites
     * the roots) must wait until the expansion has read them */
    if(!dst->ev_expand) CK(cudaEventCreateWithFlags(&dst->ev_expand, cudaEventDisableTiming));
    CK(cudaEventRecord(dst->ev_expand, dst->stream));
    CK(cudaStreamWaitEvent(src->stream, dst->ev_expand, 0));
    return POM_OK;
}

int pom_batch_apply(pom_batch* b, uint64_t env, int op, int a0, int a1, int a2)
{
    int rc = use(b); if(rc) return rc;
    if(env >= b->n_envs) return fail(POM_E_RANGE, "pom_batch_apply: env outside the batch");
    if(op < POM_OP_SPAWN_FLAME || op > POM_OP_POP_FLAME) return fail(POM_E_ARG, "pom_batch_apply: unknown op");
    if(op == POM_OP_SPAWN_FLAME && (a0 < 0 || a0 > 10 || a1 < 0 || a1 > 10 || a2 < 0 || a2 > 255))
        return fail(POM_E_ARG, "pom_batch_apply: SpawnFlame needs 0 <= x,y <= 10 and 0 <= strength <= 255");
    pomk::k_apply<<<1, 1, 0, b->stream>>>(b->recs, env, op, a0, a1, a2);
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_spawn_flame(pom_batch* b, uint64_t env, int x, int y, int strength)
{
    return pom_batch_apply(b, env, POM_OP_SPAWN_FLAME, x, y, strength);
}

int pom_make_board(int device, int32_t seed, pom_state* out, int* dirty)
{
    if(!out) return fail(POM_E_ARG, "pom_make_board: null output");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if(ce != cudaSuccess || ndev == 0) return fail(POM_E_CUDA, "no CUDA device: the step path has no CPU fallback", ce);
    if(device < 0 || device >= ndev) return fail(POM_E_ARG, "pom_make_board: no such device");
    CK(cudaSetDevice(device));
    DevBuf rec, d, aos, st;
    CK(rec.alloc(POM_REC_BYTES));
    CK(d.alloc(1));
    CK(aos.alloc(sizeof(pom_state)));
    CK(st.alloc(1));
    pomk::k_make_board<<<1, 1>>>(rec.as<uint8_t>(), d.as<uint8_t>(), seed);
    CK(cudaGetLastError());
    pomk::k_unpack<<<1, 1>>>(rec.as<uint8_t>(), aos.as<pom_state>(), st.as<uint8_t>(), 0, 1);
    CK(cudaGetLastError());
    uint8_t hd = 0;
    CK(cudaMemcpy(out, aos.p, sizeof(pom_state), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&hd, d.p, 1, cudaMemcpyDeviceToHost));
    if(dirty) *dirty = hd;
    return POM_OK;
}

int pom_batch_status(pom_batch* b, uint64_t first, uint64_t count, uint8_t* status_host)
{
    return pom_batch_download(b, first, count, nullptr, status_host);
}

int pom_batch_stats(pom_batch* b, pom_stats* out)
{
    int rc = use(b); if(rc) return rc;
    if(!out) return fail(POM_E_ARG, "pom_batch_stats: null output");
    unsigned long long h[POM_STATS_WORDS];
    CK(cudaMemcpyAsync(h, b->stats, sizeof(h), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    out->env_steps = h[pomk::ST_STEPS]; out->episodes = h[pomk::ST_EPISODES];
    for(int a = 0; a < 4; a++) out->wins[a] = h[pomk::ST_WIN0 + a];
    out->draws = h[pomk::ST_DRAWS]; out->truncated = h[pomk::ST_TRUNC];
    out->sum_episode_len = h[pomk::ST_SUMLEN]; out->invalid = h[pomk::ST_INVALID];
    return POM_OK;
}

int pom_batch_clear_stats(pom_batch* b)
{
    int rc = use(b); if(rc) return rc;
    CK(cudaMemsetAsync(b->stats, 0, POM_STATS_WORDS * sizeof(unsigned long long), b->stream));
    return POM_OK;
}

uint32_t pom_rng_moves(uint64_t seed, uint64_t env, uint32_t tick, uint32_t n_actions)
{
    return pomcore::rng_moves(seed, env, tick, n_actions);
}

int pom_batch_generate_moves(pom_batch* b, uint8_t* moves_dev, uint64_t seed, uint32_t tick, uint32_t n_actions)
{
    int rc = use(b); if(rc) return rc;
    if(!moves_dev || n_actions == 0 || n_actions > 6) return fail(POM_E_ARG, "pom_batch_generate_moves: bad argument");
    pomk::k_generate_moves<<<unsigned((b->n_envs + 255) / 256), 256, 0, b->stream>>>(
        reinterpret_cast<uint32_t*>(moves_dev), b->n_envs, b->env_offset, seed, tick, n_actions);
    b->launches++;
    CK(cudaGetLastError());
    return POM_OK;
}

uint64_t pom_batch_size(const pom_batch* b) { return b ? b->n_envs : 0; }
int      pom_batch_teams(const pom_batch* b) { return b ? (b->teams ? 1 : 0) : fail(POM_E_ARG, "pom_batch_teams: null handle"); }
int      pom_batch_radio(const pom_batch* b) { return b ? (b->radio ? 1 : 0) : fail(POM_E_ARG, "pom_batch_radio: null handle"); }

int pom_batch_records_compressed(const pom_batch* b, int* out)
{
    if(!b || !out) return fail(POM_E_ARG, "pom_batch_records_compressed: null argument");
    *out = b->recs_mapped != 0;
    return POM_OK;
}

int pom_batch_radio_download(pom_batch* b, uint64_t first, uint64_t count, uint8_t* msgs_host)
{
    int rc = use(b); if(rc) return rc;
    if(!b->radio) return fail(POM_E_ARG, "pom_batch_radio_download needs a handle made with POM_INIT_RADIO");
    if(!msgs_host) return fail(POM_E_ARG, "pom_batch_radio_download: null output");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_radio_download: range outside the batch");
    if(!count) return POM_OK;
    DevBuf buf;
    CK(buf.alloc(4 * count));
    pomk::k_radio_download<<<unsigned((count + 127) / 128), 128, 0, b->stream>>>(b->recs, buf.as<uint32_t>(), first, count);
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(msgs_host, buf.p, 4 * count, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_radio_upload(pom_batch* b, uint64_t first, uint64_t count, const uint8_t* msgs_host)
{
    int rc = use(b); if(rc) return rc;
    if(!b->radio) return fail(POM_E_ARG, "pom_batch_radio_upload needs a handle made with POM_INIT_RADIO");
    if(!msgs_host) return fail(POM_E_ARG, "pom_batch_radio_upload: null input");
    if(first > b->n_envs || count > b->n_envs - first) return fail(POM_E_RANGE, "pom_batch_radio_upload: range outside the batch");
    if(!count) return POM_OK;
    DevBuf buf;
    CK(buf.alloc(4 * count));
    CK(cudaMemcpyAsync(buf.p, msgs_host, 4 * count, cudaMemcpyHostToDevice, b->stream));
    pomk::k_radio_upload<<<unsigned((count + 127) / 128), 128, 0, b->stream>>>(b->recs, buf.as<uint32_t>(), first, count);
    b->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(b->stream));
    return POM_OK;
}

int pom_batch_set_policy_view(pom_batch* b, int view)
{
    if(!b) return fail(POM_E_ARG, "pom_batch_set_policy_view: null handle");
    b->policy_view = view;
    return POM_OK;
}

int pom_batch_get_policy_view(const pom_batch* b, int* view_out)
{
    if(!b || !view_out) return fail(POM_E_ARG, "pom_batch_get_policy_view: null argument");
    *view_out = b->policy_view;
    return POM_OK;
}
int      pom_batch_device(const pom_batch* b) { return b ? b->device : -1; }
void*    pom_batch_stream(const pom_batch* b) { return b ? (void*)b->stream : nullptr; }
void*    pom_batch_stats_device_ptr(const pom_batch* b) { return b ? (void*)b->stats : nullptr; }
void*    pom_batch_records_device_ptr(const pom_batch* b) { return b ? (void*)b->recs : nullptr; }
uint64_t pom_batch_launch_count(const pom_batch* b) { return b ? b->launches : 0; }

int pom_device_alloc(int device, uint64_t bytes, void** out)
{
    if(!out) return fail(POM_E_ARG, "pom_device_alloc: null output");
    CK(cudaSetDevice(device));
    if(cudaMalloc(out, bytes) != cudaSuccess) return fail(POM_E_NOMEM, "pom_device_alloc", cudaGetLastError());
    return POM_OK;
}

int pom_device_free(int device, void* p)
{
    CK(cudaSetDevice(device));
    CK(cudaFree(p));
    return POM_OK;
}

int pom_host_alloc(uint64_t bytes, void** out)
{
    if(!out) return fail(POM_E_ARG, "pom_host_alloc: null output");
    /* page-locked for every device of the process and mapped into their address spaces (zero-copy step_host) */
    if(cudaHostAlloc(out, bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) return fail(POM_E_NOMEM, "pom_host_alloc", cudaGetLastError());
    return POM_OK;
}

int pom_bind_thread_near(int device)
{
    cpu_set_t set;
    if(local_cpus(device, &set)) sched_setaffinity(0, sizeof(set), &set);
    return POM_OK;
}

int pom_host_alloc_near(int device, uint64_t bytes, void** out)
{
    if(!out) return fail(POM_E_ARG, "pom_host_alloc_near: null output");
    cpu_set_t before, near;
    const bool have_before = sched_getaffinity(0, sizeof(before), &before) == 0;
    const bool moved = have_before && local_cpus(device, &near) && sched_setaffinity(0, sizeof(near), &near) == 0;
    /* the pages are allocated and first touched (pinning touches them) by this thread, now running next to the GPU */
    const int rc = pom_host_alloc(bytes, out);
    if(rc == POM_OK) std::memset(*out, 0, bytes);
    if(moved) sched_setaffinity(0, sizeof(before), &before);
    return rc;
}

int pom_host_free(void* p)
{
    CK(cudaFreeHost(p));
    return POM_OK;
}

int pom_batch_event_record(pom_batch* b, int which)
{
    int rc = use(b); if(rc) return rc;
    if(which < 0 || which > 1) return fail(POM_E_ARG, "pom_batch_event_record: which must be 0 or 1");
    CK(cudaEventRecord(b->ev[which], b->stream));
    return POM_OK;
}

int pom_batch_event_elapsed_ms(pom_batch* b, float* ms)
{
    int rc = use(b); if(rc) return rc;
    if(!ms) return fail(POM_E_ARG, "pom_batch_event_elapsed_ms: null output");
    CK(cudaEventSynchronize(b->ev[1]));
    CK(cudaEventElapsedTime(ms, b->ev[0], b->ev[1]));
    return POM_OK;
}

int pom_batch_flush_l2(pom_batch* b)
{
    int rc = use(b); if(rc) return rc;
    if(!b->flush_buf) CK(cudaMalloc(&b->flush_buf, FLUSH_BYTES));
    const uint64_t n16 = FLUSH_BYTES / 16;
    pomk::k_fill_zero<<<unsigned((n16 + 255) / 256), 256, 0, b->stream>>>(reinterpret_cast<uint4*>(b->flush_buf), n16);
    CK(cudaGetLastError());
    return POM_OK;
}

}
