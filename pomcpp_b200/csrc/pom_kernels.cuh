/*
 * pom_kernels.cuh — sm_100a kernels of the batched step path.
 *
 *  K1 k_step_ws     per-tick mode, persistent and warp-specialised: one CTA per SM, a ring of 24 slice buffers in shared
 *                   memory (32 consecutive 292-byte records + the slice's move bytes each), a producer warp that keeps
 *                   them filled with 1-D TMA bulk copies (cp.async.bulk + mbarrier), 20 compute warps that run the tick
 *                   (pom_core.cuh) in place and bulk-store the slice.  HBM traffic per env-step = 292 B in + 292 B out +
 *                   4 B of moves (2 B as a joint action); no thread issues a global load/store for state.  The record
 *                   stride of 73 words is odd, so same-field accesses of the 32 lanes are bank-conflict free.
 *     k_step        round 1's form (one CTA per tile, every warp loads -> ticks -> stores its own slice), kept as
 *                   POM_STEP_KERNEL=tile and as the oracle of test_persistent_kernel_equals_tile_kernel.
 *  K2 k_rollout     fused K-tick mode: per-warp staging once, then K ticks on the resident record with actions
 *                   from the stateless counter RNG (or the caller's tick-major moves), truncation, episode statistics
 *                   and auto-reset from the template pool inside the kernel.
 *  K3 k_make_templates / k_fill_from_templates   board generation on the device and env (re)initialisation.
 *  K4 k_gather_records / k_expand_step           state copy (pom_batch_clone) and tree-search fan-out (+ one Step, fused).
 *  K5 k_pack / k_unpack / k_observe              AoS bboard::State <-> packed record; the State as one agent sees it (fog).
 *     k_observe_planes                            the same view as byte planes for a network input, four lanes per env.
 *  K7 k_policy_moves / k_rollout<TPB, true>   the reference's SimpleAgent (pom_policy.cuh) as the action source: per tick
 *                                                 into a moves buffer, or inside the fused rollout; the agents' 8-byte
 *                                                 memories live in global memory, word-major (coalesced, L1/L2-resident).
 *  K6 stats                                      episode counters gathered per lane in registers, one warp reduction and
 *                                                 one atomicAdd per counter, warp and launch; warp-cooperative reset (cp.async).
 */
#ifndef POM_KERNELS_CUH_
#define POM_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>
#include "pom_core.cuh"
#include "pom_policy.cuh"
#include "pom_batch.h"

namespace pomk
{

/* internal flag of the per-tick kernels (not part of the ABI): envs whose status carries TRUNCATED are frozen too, as in
 * the fused rollout (pom_batch_rollout run tick by tick) */
constexpr uint32_t STEP_FREEZE_TRUNCATED = 0x40000000u;

enum { ST_STEPS = 0, ST_EPISODES = 1, ST_WIN0 = 2, ST_DRAWS = 6, ST_TRUNC = 7, ST_SUMLEN = 8, ST_INVALID = 9 };

struct BatchParams {
    uint8_t*            recs;         /* n_envs packed records, allocated in whole 256-env tiles */
    uint64_t            n_envs;
    uint64_t            env_offset;   /* global index of env 0                                   */
    const uint8_t*      templates;    /* n_templates packed records                              */
    uint32_t            n_templates;
    uint32_t            tmpl_mask;    /* n_templates - 1 when that is a power of two (template index without a division), else 0 */
    uint32_t            max_ticks;
    uint32_t*           episodes;     /* per-env number of finished episodes                     */
    unsigned long long* stats;        /* POM_STATS_WORDS counters                                */
    uint32_t*           policy;       /* SimpleAgent memories, SoA: word k of env e at [k * policy_stride + e], k = 2*agent + {0,1}
                                         (the two words of pom_simple_agent); k = 8: the episode number they belong to.
                                         Null until a policy entry point is used. */
    uint64_t            policy_stride;
};

/* ---------------------------------------------------------------- TMA 1-D bulk copy + mbarrier (PTX) */
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
/* global -> shared, completion signalled on the mbarrier (SASS: UBLKCP) */
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
/* shared -> global, tracked by a bulk async-group */
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read_all()
{
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

/* ---------------------------------------------------------------- K6: episode statistics */
__device__ __forceinline__ void warp_add(unsigned long long* dst, uint32_t v)
{
    const uint32_t s = __reduce_add_sync(0xFFFFFFFFu, v);
    if((threadIdx.x & 31u) == 0u && s) atomicAdd(dst, (unsigned long long)s);
}

/* Episode statistics are gathered per lane in registers (16-bit counters, two to a word) and added to the global
 * counters ONCE per warp and launch (acc_flush): one warp reduction and one atomicAdd per counter, instead of three
 * reductions and up to nine atomics in every tick in which some env of the warp finished (1.3 M warp-instructions per
 * 1 Mi-env tick, profiles/k_step_by_function_r2.txt). */
struct EpisodeAcc {
    uint32_t fin_draw = 0u;      /* episodes | draws << 16      */
    uint32_t trunc_abort = 0u;   /* truncated | aborted << 16   */
    uint32_t win01 = 0u, win23 = 0u;
    uint32_t len = 0u;           /* sum of episode lengths      */
    uint32_t steps = 0u;         /* env-steps executed          */
    uint32_t pending = 0u;       /* episodes since the last flush (16-bit counters: flush before 65536) */
};

__device__ __forceinline__ void acc_add(EpisodeAcc& A, bool fin, uint32_t status, uint32_t len)
{
    if(!fin) return;
    /* exactly one outcome per episode: DONE (won | draw) > TRUNCATED > aborted (left the reference's domain) */
    const bool done = (status & POM_STATUS_DONE) != 0u;
    const bool draw = done && (status & POM_STATUS_DRAW);
    const bool trunc = !done && (status & POM_STATUS_TRUNCATED);
    const uint32_t w = (status & POM_STATUS_WINNER_MASK) >> POM_STATUS_WINNER_SHIFT;
    A.fin_draw += 1u + (draw ? 0x10000u : 0u);
    A.trunc_abort += (trunc ? 1u : 0u) + ((!done && !trunc) ? 0x10000u : 0u);
    if(done && !draw)
    {
        const uint32_t inc = (w & 1u) ? 0x10000u : 1u;
        if(w & 2u) A.win23 += inc; else A.win01 += inc;
    }
    A.len += len;
    A.pending++;
}

/* called by ALL 32 lanes */
__device__ __forceinline__ void acc_flush(unsigned long long* stats, EpisodeAcc& A, bool count_steps)
{
    const uint32_t lane = threadIdx.x & 31u;
    if(__reduce_or_sync(0xFFFFFFFFu, A.pending))
    {
        const uint32_t v[9] = { A.fin_draw & 0xFFFFu, A.win01 & 0xFFFFu, A.win01 >> 16, A.win23 & 0xFFFFu, A.win23 >> 16,
                                A.fin_draw >> 16, A.trunc_abort & 0xFFFFu, A.len, A.trunc_abort >> 16 };
        /* ST_EPISODES = 1, ST_WIN0..3 = 2..5, ST_DRAWS = 6, ST_TRUNC = 7, ST_SUMLEN = 8, ST_INVALID = 9 */
#pragma unroll
        for(int k = 0; k < 9; k++)
        {
            const uint32_t sum = __reduce_add_sync(0xFFFFFFFFu, v[k]);
            if(lane == 0u && sum) atomicAdd(stats + 1 + k, (unsigned long long)sum);
        }
    }
    if(count_steps)
    {
        const uint32_t sum = __reduce_add_sync(0xFFFFFFFFu, A.steps);
        if(lane == 0u && sum) atomicAdd(stats + ST_STEPS, (unsigned long long)sum);
    }
    A = EpisodeAcc();
}

/* end-of-tick episode handling shared by K1 (auto-reset flag) and K2: truncate, count, reset.
 * Must be called by all 32 lanes of a warp.  The reset is warp-cooperative: for every lane whose env
 * finished, all 32 lanes copy that env's template record (73 words) into shared memory, instead of one
 * lane running a 73-iteration loop while 31 lanes wait.  `warp_recs` = the warp's 32 consecutive records. */
__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gmem_src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.wait_all;" ::: "memory");
}

/* `ep_now` = this env's episode number, loaded by the caller at kernel start (one coalesced load) so that
 * the reset path does not expose a dependent global load.  Returns the env's end-of-tick status byte as it was
 * BEFORE a reset (what an RL loop needs to see: done / winner / truncated of the episode that just ended). */
__device__ __forceinline__ uint32_t finish_and_reset(uint8_t* warp_recs, uint8_t* rec, const BatchParams& P, uint64_t env, bool active, bool do_reset,
                                                 uint32_t& ep_now, EpisodeAcc& acc)
{
    uint32_t st = active ? rec[R_STATUS] : 0u;
    const uint32_t len = active ? *reinterpret_cast<const uint16_t*>(rec + R_TIME) : 0u;
    if(active && !(st & POM_STATUS_DONE) && P.max_ticks && len >= P.max_ticks) st |= POM_STATUS_TRUNCATED;
    const bool fin = active && (st & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID)) != 0u;
    uint32_t pending = __ballot_sync(0xFFFFFFFFu, fin);
    if(pending == 0u) return st;
    acc_add(acc, fin, st, len);
    if(!do_reset)
    {
        if(fin) rec[R_STATUS] = uint8_t(st);
        return st;
    }
    uint32_t tmpl = 0u;
    if(fin)
    {
        const uint32_t ep = ++ep_now;
        P.episodes[env] = ep;
        /* (env_offset + env + ep) % n_templates without 64-bit division on the common path */
        const uint64_t g = P.env_offset + env + ep;
        tmpl = P.tmpl_mask ? (uint32_t(g) & P.tmpl_mask) : (g < 0xFFFFFFFFull ? uint32_t(g) % P.n_templates : uint32_t(g % P.n_templates));
    }
    const uint32_t lane = threadIdx.x & 31u;
    while(pending)
    {
        const uint32_t src_lane = uint32_t(__ffs(int(pending))) - 1u;
        pending &= pending - 1u;
        const uint32_t t = __shfl_sync(0xFFFFFFFFu, tmpl, int(src_lane));
        const uint32_t* src = reinterpret_cast<const uint32_t*>(P.templates) + size_t(t) * POM_REC_WORDS;
        uint32_t* dst = reinterpret_cast<uint32_t*>(warp_recs + size_t(src_lane) * POM_REC_BYTES);
        /* asynchronous global->shared copies: the templates of all finished lanes are in flight together */
        cp_async_4(dst + lane, src + lane);
        cp_async_4(dst + lane + 32u, src + lane + 32u);
        if(lane < uint32_t(POM_REC_WORDS - 64)) cp_async_4(dst + lane + 64u, src + lane + 64u);
    }
    cp_async_wait_all();
    __syncwarp();
    return st;
}

/* ---------------------------------------------------------------- one tick of the warp's 32 envs */
/* The tick runs one env per lane (pom_core.cuh) except for its two rare, long, divergent pieces: the flame pops at the
 * start (TickFlames -> PopFlame) and the explosions at the end (TickBombs -> ExplodeTopBomb -> SpawnFlame).  An env
 * needs them in 11 % / 16 % of its ticks, so with one env per lane nearly every warp ran them with 2-3 of 32 lanes
 * active (profiles/k_step_by_function_r1.txt).  Here the warp votes which envs are due (__ballot_sync), and every
 * group of four lanes takes one due env, one lane per ray / arm: flame reach is resolved by four lanes walking the
 * four rays at once, the kills and the chain test are combined with __shfl_xor_sync inside the group. */
constexpr uint32_t FULL_WARP = 0xFFFFFFFFu;

/* Which env does group `quad` serve this round?  The due lanes write their lane index into an 8-byte list in shared
 * memory at the position of their rank among the due lanes (ranks 8.. wait for the next round); group q reads entry q.
 * Returns 32 when the group has nothing to do.  `wlist`: 8 bytes of shared memory owned by this warp. */
__device__ __forceinline__ uint32_t due_env_of_group(uint8_t* wlist, uint32_t mask, bool due, uint32_t lane, uint32_t quad, uint32_t& rank)
{
    rank = uint32_t(__popc(mask & ((1u << lane) - 1u)));
    if(due && rank < 8u) wlist[rank] = uint8_t(lane);
    __syncwarp();
    const uint32_t e = quad < uint32_t(__popc(mask)) ? wlist[quad] : 32u;
    __syncwarp();                                             /* the list is rewritten next round */
    return e;
}

/* the pop loop of util::TickFlames (step_utility.cpp:216-222); `due` = this lane's front flame has expired.
 * Called by all 32 lanes. */
__device__ __forceinline__ void warp_pop_due(uint8_t* sslice, const uint8_t* rec, bool due, uint8_t* wlist)
{
    const uint32_t lane = threadIdx.x & 31u, quad = lane >> 2, arm = lane & 3u;
    int turns = due ? int(rec[R_FCOUNT]) : 0;                 /* flameCount turns at most */
    for(;;)
    {
        const uint32_t mask = __ballot_sync(FULL_WARP, due);
        if(mask == 0u) break;
        uint32_t rank;
        const uint32_t e = due_env_of_group(wlist, mask, due, lane, quad, rank);
        uint8_t* r = sslice + e * POM_REC_BYTES;
        if(e < 32u) pomcore::pop_flame_arm(r, arm);
        __syncwarp();                                         /* every arm has read the front entry */
        if(e < 32u && arm == 0u) pomcore::pop_flame_ring(r);
        __syncwarp();
        if(due && rank < 8u)
        {
            turns--;
            due = turns > 0 && rec[R_FTIME + rec[R_FINDEX]] == 0;
        }
    }
}

/* the explosion loop of util::TickBombs (step_utility.cpp:231-244); `due` = this lane's bombs[0] has timed out.
 * Called by all 32 lanes.  A group scans its four rays without writing; if no ray meets a bomb the rays are committed
 * and lane 0 of the group does the rest of ExplodeTopBomb; else the env's own lane runs the serial machine. */
__device__ __forceinline__ void warp_explode_due(uint8_t* sslice, uint8_t* rec, bool due, int& flags, uint8_t* wlist)
{
    const uint32_t lane = threadIdx.x & 31u, quad = lane >> 2, ray = lane & 3u;
    int turns = due ? int(rec[R_BCOUNT]) : 0;                 /* bombCount turns at most */
    for(;;)
    {
        const uint32_t mask = __ballot_sync(FULL_WARP, due);
        if(mask == 0u) break;
        uint32_t rank;
        const uint32_t e = due_env_of_group(wlist, mask, due, lane, quad, rank);
        uint8_t* r = sslice + e * POM_REC_BYTES;
        uint32_t plan = 0u, ci0 = 0u, slot = 0u, c = 0u;
        int stride = 0;
        if(e < 32u)
        {
            c = pomcore::bomb_slot(r, r[R_BINDEX]);
            const uint32_t p = c & 0xFFu;
            ci0 = uint32_t(pomcore::cell_of(p));
            slot = pomcore::ring20(uint32_t(r[R_FINDEX]) + r[R_FCOUNT]);
            const uint32_t len = pomcore::ray_length(p, (c >> 12) & 15u, ray, stride);
            plan = pomcore::ray_scan(r, ci0, stride, len);
        }
        uint32_t all = plan | __shfl_xor_sync(FULL_WARP, plan, 1);
        all |= __shfl_xor_sync(FULL_WARP, all, 2);
        const bool chain = (all & pomcore::RAY_CHAIN) != 0u;
        __syncwarp();                                         /* all four lanes have read the top bomb and the flame ring */
        if(e < 32u && !chain)
        {
            pomcore::ray_commit(r, ci0, stride, plan, slot);  /* rays and origin are disjoint cells */
            /* the rest of ExplodeTopBomb, shared out: lane 0 the flame entry and the origin cell, lane 1 the kills,
             * lane 2 PopBomb (three disjoint sets of fields) */
            if(pomcore::top_bomb_commit_part(r, c, all, ray, slot)) r[R_STATUS] |= POM_STATUS_INVALID;
        }
        const uint32_t chained = __ballot_sync(FULL_WARP, chain);   /* bit 4q: the explosion served by group q chains */
        __syncwarp();                                         /* the groups' writes are visible to the envs' own lanes */
        if(due && rank < 8u)
        {
            if((chained >> (4u * rank)) & 1u)
            {
                flags |= pomcore::step_explode_due(rec);      /* finishes the loop for this env */
                due = false;
            }
            else
            {
                turns--;
                due = turns > 0 && pomcore::top_bomb_due(rec);
            }
        }
        __syncwarp();
    }
}

/* bboard::Step (+ Environment::Step's bookkeeping unless raw; TEAMS: the team game's, pomcore::env_post) for the env of
 * every lane with `step` set */
template<bool TEAMS = false>
__device__ __forceinline__ void warp_tick(uint8_t* sslice, uint8_t* rec, uint32_t m, bool step, bool raw, uint8_t* wlist,
                                          int invalid_mask = pomcore::F_INVALID_MASK)
{
    const bool pops = step && pomcore::flames_age(rec);       /* TickFlames, step.cpp:15 */
    warp_pop_due(sslice, rec, pops, wlist);
    int flags = 0;
    bool due = false;
    if(step) flags = pomcore::step_body(rec, m, due, false);
    warp_explode_due(sslice, rec, due, flags, wlist);
    if(step)
    {
        if(flags & invalid_mask) rec[R_STATUS] |= POM_STATUS_INVALID;
        if(!raw) pomcore::env_post<TEAMS>(rec);
    }
}

/* observation planes of agent `agent` for the warp's 32 resident records: every quad of lanes writes the observations
 * of four envs (quad q: envs q, q + 8, q + 16, q + 24 of the slice), lane i of the quad the chunks i, i + 4, i + 8, i + 12
 * (pomcore::observe_part_chunks), so that every store instruction of the warp covers eight full 128-byte lines.
 * `out0` = the observation of the slice's first env, `n_valid` = envs of the slice inside the batch.  All 32 lanes call. */
/* the cropped layout (pomcore::observe_cropped_part_*): records of `rec_bytes`; every lane patches its own flame cells */
__device__ __forceinline__ void warp_observe_slice_cropped(const uint8_t* sslice, int agent, int view, uint8_t* out0, uint32_t n_valid, uint32_t rec_bytes)
{
    const uint32_t lane = threadIdx.x & 31u, quad = lane >> 2;
    const int part = int(lane & 3u);
#pragma unroll 1
    for(uint32_t m = 0; m < 4u; m++)
    {
        const uint32_t e = quad + 8u * m;
        const bool valid = e < n_valid;
        const uint8_t* r = sslice + e * POM_REC_BYTES;
        uint8_t* out = out0 + size_t(e) * rec_bytes;
        uint32_t flames = 0u;
        if(valid) flames = pomcore::observe_cropped_part_chunks(r, agent, view, out, part);
        __syncwarp();                                         /* the quad's chunk stores are ordered before its patches */
        if(valid) pomcore::observe_cropped_part_patches(r, agent, view, out, part, flames);
    }
}

__device__ __forceinline__ void warp_observe_slice(const uint8_t* sslice, int agent, int view, uint8_t* out0, uint32_t n_valid)
{
    const uint32_t lane = threadIdx.x & 31u, quad = lane >> 2;
    const int part = int(lane & 3u);
#pragma unroll 1
    for(uint32_t m = 0; m < 4u; m++)
    {
        const uint32_t e = quad + 8u * m;
        const bool valid = e < n_valid;
        const uint8_t* r = sslice + e * POM_REC_BYTES;
        uint8_t* out = out0 + size_t(e) * POM_OBS_BYTES;
        pomcore::ObsWindow W{};
        uint32_t lit = 0u;
        if(valid)
        {
            W = pomcore::obs_window(r, agent, view);
            lit = pomcore::observe_part_chunks(r, agent, W, out, part);
        }
        lit |= __shfl_xor_sync(FULL_WARP, lit, 1);
        lit |= __shfl_xor_sync(FULL_WARP, lit, 2);
        __syncwarp();                                         /* the quad's chunk stores are ordered before its patches */
        if(valid) pomcore::observe_part_patches(r, W, out, part, lit);
    }
}

/* dynamic shared memory of the tile kernels: TPB records + one mbarrier per warp */
template<int TPB> struct TileScratch {
    static constexpr uint32_t OFF_BAR = TPB * POM_REC_BYTES;
    static constexpr uint32_t OFF_LIST = OFF_BAR + 64;        /* 8 bytes per warp: due_env_of_group */
    static constexpr uint32_t BYTES = OFF_LIST + 8 * (TPB / 32);
};

/* ---------------------------------------------------------------- K1: per-tick kernel */
/* TEAMS (here and in every kernel below that takes it): the 2v2 team game - its episode rule (pomcore::env_post) and its
 * SimpleAgent (pompolicy::plan_agent).  The mode belongs to the handle; the free-for-all images are the default. */
template<int TPB, bool TEAMS = false>
__global__ void __launch_bounds__(TPB) k_step(BatchParams P, const uint32_t* __restrict__ moves, uint32_t flags, uint8_t* __restrict__ status_out)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const uint64_t env = uint64_t(blockIdx.x) * TPB + threadIdx.x;
    const bool active = env < P.n_envs;
    const bool raw = (flags & POM_STEP_RAW) != 0u;

    /* Warp-independent staging: every warp bulk-loads, steps and bulk-stores its own 32-record slice
     * (9344 bytes) behind its own mbarrier.  No CTA-wide barrier: a warp whose 32 envs had a quiet tick
     * does not wait for a warp that had to run a chain explosion. */
    constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + TileScratch<TPB>::OFF_BAR) + warp;
    uint8_t* sslice = smem + warp * SLICE_BYTES;
    uint8_t* gslice = P.recs + (size_t(blockIdx.x) * TPB + warp * 32u) * POM_REC_BYTES;
    if(lane == 0)
    {
        mbar_init(bar, 1);
        fence_barrier_init();
        mbar_expect_tx(bar, SLICE_BYTES);
        bulk_g2s(sslice, gslice, SLICE_BYTES, bar);
    }
    const uint32_t m = active ? __ldg(moves + env) : 0u;     /* both loads overlap the bulk load */
    uint32_t ep_now = (active && (flags & POM_STEP_AUTORESET)) ? P.episodes[env] : 0u;
    __syncwarp();
    mbar_wait(bar, 0);

    uint8_t* rec = sslice + lane * POM_REC_BYTES;
    /* finished envs are skipped (environment.cpp:125) unless raw; invalid envs always freeze */
    const bool stepped = active && !(rec[R_STATUS] & (raw ? POM_STATUS_INVALID : (POM_STATUS_DONE | POM_STATUS_INVALID)));
    warp_tick<TEAMS>(sslice, rec, m, stepped, raw, smem + TileScratch<TPB>::OFF_LIST + 8u * warp,
                     (flags & POM_STEP_CONTINUE_UNDEFINED) ? pomcore::F_INVALID_MASK_CONTINUE : pomcore::F_INVALID_MASK);
    EpisodeAcc acc;
    acc.steps = stepped ? 1u : 0u;
    uint32_t st_end = active ? rec[R_STATUS] : 0u;
    if(flags & POM_STEP_AUTORESET)
    {
        const uint32_t st = finish_and_reset(sslice, rec, P, env, active && stepped, true, ep_now, acc);
        if(active && stepped) st_end = st;
    }
    acc_flush(P.stats, acc, (flags & POM_STEP_COUNT) != 0u);
    if(status_out && active) status_out[env] = uint8_t(st_end);   /* one coalesced byte per env */
    fence_proxy_async();                                      /* generic-proxy writes -> visible to the bulk store */
    __syncwarp();
    if(lane == 0)
    {
        bulk_s2g(gslice, sslice, SLICE_BYTES);
        bulk_wait_read_all();                                 /* smem must stay valid until it has been read */
    }
}

/* ---------------------------------------------------------------- K1, persistent form: k_step_ws */
/* One CTA per SM for the whole launch.  Shared memory is a ring of NBUF slice buffers (32 records + the slice's 32 x 4
 * move bytes each); warp NW is the PRODUCER: it keeps every free buffer filled with the CTA's next slice (TMA bulk load,
 * completion on the buffer's `full` mbarrier).  Warps 0..NW-1 COMPUTE: a warp takes the next ticket (shared-memory
 * counter), reads from the ticket's mail slot which buffer its slice is landing in, waits for that buffer's `full`
 * barrier, runs the tick on it in place, bulk-stores it and returns the buffer to the free mask once the store has read
 * it.  NBUF > NW, so NBUF - NW loads are always in flight ahead of the compute warps, and nothing is relaunched or
 * drained between slices.
 * With k_step every warp did load -> tick -> store itself; once the tick got cheap (vectorised movement, shared-out
 * explosions) ncu showed 4 long-scoreboard stall cycles per issue and 45 % issue utilisation: the 24 resident warps
 * spent 40 % of their time waiting for their own loads (profiles/k_step_ncu_summary_r2b.json).
 * Slices are dealt round-robin over the CTAs (slice = blockIdx.x + ticket * gridDim.x): at any time the CTAs work on a
 * window of neighbouring slices, and a warp knows its slice from its ticket alone. */
/* inputs and outputs of one per-tick launch besides the records */
struct StepIO {
    const void* moves;         /* n_envs x 4 move bytes (uint32 per env), or n_envs joint actions (uint16 per env) when joint != 0 */
    uint32_t    joint;         /* j = a0 + 6 a1 + 36 a2 + 216 a3 (the encoding of pom_batch_expand_step) */
    uint32_t    bulk;          /* moves are 16-byte aligned: fetch them with the slice's TMA load */
    uint32_t    reverse;       /* walk the batch from its last slice to its first.  The host alternates the direction tick by
                                  tick: a tick then STARTS with the records the previous tick touched last, which are still in
                                  the 126 MB L2 (read hits, and their write-backs are merged with this tick's stores) */
    uint8_t*    status_out;    /* one end-of-tick status byte per env, or null */
    uint32_t*   done_bits;     /* one word per slice: bit l = env 32 s + l ended an episode this tick, or null */
    uint32_t*   fin_env;       /* compacted list of those envs ...            (null: no list) */
    uint8_t*    fin_status;    /* ... and their status bytes (as in status_out) */
    uint32_t*   fin_counter;   /* DEVICE words: [0] the counter the list is appended through, [1] CTAs that are done */
    uint32_t*   fin_count_out; /* where the last CTA publishes the list length (device or mapped host memory) */
    uint32_t    fin_capacity;
    uint8_t*    obs;           /* observation planes of the agents in obs_mask, written from the resident record at the
                                  end of the tick (after an auto-reset): slab k (k-th agent of the mask) at
                                  obs + k * obs_stride * POM_OBS_BYTES; null = none.
                                  The REWARDS images, which are OBS = false images, take their output here instead:
                                  one word per env, byte a = the int8 reward of agent a (pomcore::tick_rewards).  The slot
                                  keeps its one type: a union with a uint32_t* changed the SASS of the OBS images. */
    uint64_t    obs_stride;
    uint32_t    obs_mask;
    int         obs_view;
};
/* the kernel-parameter size is part of every k_step_ws image: a new output shares a slot instead of growing the struct */
static_assert(sizeof(StepIO) == 104, "StepIO changes the parameter block of every k_step_ws image");

/* four moves from a joint action index */
__device__ __forceinline__ uint32_t moves_of_joint(uint32_t j)
{
    const uint32_t a0 = j % 6u, r1 = j / 6u, a1 = r1 % 6u, r2 = r1 / 6u, a2 = r2 % 6u, a3 = (r2 / 6u) % 6u;
    return a0 | (a1 << 8) | (a2 << 16) | (a3 << 24);
}

template<int NBUF> struct RingScratch {
    static constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    static constexpr uint32_t SLOT = SLICE_BYTES + 128 + 16;      /* records, the slice's moves, the warp's due list */
    static constexpr uint32_t OFF_FULL = NBUF * SLOT;
    /* mail[t % MAIL]: which buffer holds the slice of ticket t, written by the producer: (t + 1) << 8 | buffer << 1 |
     * phase parity of the buffer's `full` barrier */
    static constexpr uint32_t MAIL = 256;
    static constexpr uint32_t OFF_MAIL = OFF_FULL + 8 * NBUF;
    static constexpr uint32_t OFF_TICKET = OFF_MAIL + 4 * MAIL;    /* [0] next ticket, [1] warps done, [2] free-buffer mask */
    /* finished-env list of this CTA, handed to the global list in one piece when the CTA is done: word [0] = entries
     * reserved, word [1] = position of the first reservation that did not fit (0xFFFFFFFF: all fit) */
    static constexpr uint32_t FIN_CAP = 480;
    static constexpr uint32_t OFF_FIN = OFF_TICKET + 16;
    static constexpr uint32_t OFF_FIN_ENV = OFF_FIN + 16;
    static constexpr uint32_t OFF_FIN_ST = OFF_FIN_ENV + 4 * FIN_CAP;
    static constexpr uint32_t BYTES = OFF_FIN_ST + FIN_CAP;
};

/* OBS: the kernel image with the observation code (StepIO::obs); the plain step runs the image without it - 1200
 * instructions less in the loop body of a kernel whose warps are spread all over the instruction cache */
/* FREEZE: envs whose status carries TRUNCATED are frozen too, as in the fused rollout (pom_batch_rollout run tick by tick) */
/* SPEC: the image of the plain actor / bench loop - flags == AUTORESET | COUNT, four move bytes per env fetched with
 * the slice, no per-env outputs - with everything a launch parameter would decide known at compile time: the generic
 * image tests flags and pointers inside the loop body, and specialised a tick is 3-4 % faster (0.1052 -> 0.1008 ms with
 * the two-stream overlap).  The same treatment of the compact-I/O configuration was measured 6-15 % SLOWER than the
 * generic image in three variants (all of io constant; the flags only; joint + bulk only) and is not built: what the
 * compiler makes of this loop body is not monotone in what it knows (see also FREEZE below). */
/* REWARDS: the image of pom_batch_step_rewards - every active env also stores its four int8 rewards (pomcore::tick_rewards)
 * as one word to the array in StepIO::obs, next to its status byte.  Its own image for the reason FREEZE and TEAMS have theirs:
 * the plain step keeps its code as it is. */
template<int NW, int NBUF, bool OBS, bool FREEZE, bool SPEC = false, bool TEAMS = false, bool REWARDS = false>
__global__ void __launch_bounds__((NW + 1) * 32, 1) k_step_ws(BatchParams P, StepIO io_in, uint32_t flags_in)
{
    const uint32_t flags = SPEC ? uint32_t(POM_STEP_AUTORESET | POM_STEP_COUNT) : flags_in;
    StepIO io = io_in;
    if(SPEC)
    {
        io.joint = 0u; io.bulk = 1u; io.status_out = nullptr; io.obs = nullptr; io.done_bits = nullptr; io.fin_env = nullptr;
    }
    const uint32_t* __restrict__ moves = static_cast<const uint32_t*>(io.moves);
    const uint16_t* __restrict__ joint = static_cast<const uint16_t*>(io.moves);
    uint8_t* __restrict__ status_out = io.status_out;
    const uint32_t moves_bulk = io.bulk;
    const uint32_t mv_bytes = io.joint ? 64u : 128u;              /* move bytes per slice */
    extern __shared__ __align__(128) uint8_t smem[];
    typedef RingScratch<NBUF> R;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + R::OFF_FULL);
    volatile uint32_t* mail = reinterpret_cast<volatile uint32_t*>(smem + R::OFF_MAIL);
    uint32_t* ticket = reinterpret_cast<uint32_t*>(smem + R::OFF_TICKET);
    uint32_t* free_mask = ticket + 2;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint64_t n_slices = (P.n_envs + 31u) / 32u;
    /* this CTA's slices: blockIdx.x, blockIdx.x + gridDim.x, ... */
    const uint32_t T = blockIdx.x < n_slices ? uint32_t((n_slices - blockIdx.x + gridDim.x - 1u) / gridDim.x) : 0u;
    if(threadIdx.x == 0)
    {
        for(int b = 0; b < NBUF; b++) mbar_init(full + b, 1);
        ticket[0] = 0u;
        ticket[1] = 0u;                                               /* compute warps that have finished */
        *free_mask = (NBUF >= 32) ? 0xFFFFFFFFu : ((1u << NBUF) - 1u);
        reinterpret_cast<uint32_t*>(smem + R::OFF_FIN)[0] = 0u;
        reinterpret_cast<uint32_t*>(smem + R::OFF_FIN)[1] = 0xFFFFFFFFu;
        fence_barrier_init();
    }
    for(uint32_t i = threadIdx.x; i < R::MAIL; i += blockDim.x) mail[i] = 0u;
    __syncthreads();

    if(warp == NW)
    {
        /* PRODUCER.  Buffers are handed out from a free mask, not in ring order: a slice that takes long (a chained
         * explosion, many resets) keeps its own buffer busy and nothing else - with an in-order ring everything 24
         * tickets behind it waited (15 % of the compute warps' time, profiles/k_step_ncu_summary_r2.json). */
        if(lane != 0) return;
        uint32_t parity = 0u;                                         /* bit b: phase parity of full[b]'s next use */
        for(uint32_t t = 0; t < T; t++)
        {
            uint32_t fm;
            while((fm = *reinterpret_cast<volatile uint32_t*>(free_mask)) == 0u) __nanosleep(40);
            const uint32_t b = uint32_t(__ffs(int(fm))) - 1u;
            atomicAnd(free_mask, ~(1u << b));
            const uint64_t s0 = blockIdx.x + uint64_t(t) * gridDim.x;
            const uint64_t s = io.reverse ? n_slices - 1u - s0 : s0;
            const bool whole = (s + 1u) * 32u <= P.n_envs;                /* the last slice's moves may end early: per-lane loads */
            const uint32_t mbytes = (moves_bulk && whole) ? mv_bytes : 0u;
            mbar_expect_tx(full + b, R::SLICE_BYTES + mbytes);
            bulk_g2s(smem + b * R::SLOT, P.recs + s * R::SLICE_BYTES, R::SLICE_BYTES, full + b);
            if(mbytes) bulk_g2s(smem + b * R::SLOT + R::SLICE_BYTES, static_cast<const uint8_t*>(io.moves) + s * mv_bytes, mbytes, full + b);
            /* tell the warp that holds (or will hold) ticket t where its slice lands.  The buffer was free, so its
             * previous load had completed: `full[b]` is in the phase this load completes - a parity wait on it cannot
             * mistake an older phase for this one. */
            mail[t % R::MAIL] = ((t + 1u) << 8) | (b << 1) | ((parity >> b) & 1u);
            parity ^= 1u << b;
        }
        return;
    }

    const bool raw = (flags & POM_STEP_RAW) != 0u;
    EpisodeAcc acc;
    for(;;)
    {
        uint32_t t = 0u;
        if(lane == 0) t = atomicAdd(ticket, 1u);
        t = __shfl_sync(FULL_WARP, t, 0);
        if(t >= T) break;
        const uint64_t s0 = blockIdx.x + uint64_t(t) * gridDim.x;
        const uint64_t s = io.reverse ? n_slices - 1u - s0 : s0;
        const uint64_t env = s * 32u + lane;
        const bool active = env < P.n_envs;
        const bool whole = (s + 1u) * 32u <= P.n_envs;
        uint32_t m = 0u;
        if(!(moves_bulk && whole) && active) m = io.joint ? uint32_t(__ldg(joint + env)) : __ldg(moves + env);   /* overlaps the wait below */
        uint32_t ep_now = (active && (flags & POM_STEP_AUTORESET)) ? P.episodes[env] : 0u;
        /* where is my slice?  (The mail slot of ticket t is rewritten for ticket t + 256; by then this warp has long read
         * it: the producer is never more than the 24 buffers ahead of the warps.) */
        uint32_t v;
        while(((v = mail[t % R::MAIL]) >> 8) != t + 1u) __nanosleep(20);
        const uint32_t b = (v >> 1) & 31u;
        uint8_t* sslice = smem + b * R::SLOT;
        mbar_wait(full + b, v & 1u);
        if(moves_bulk && whole)
            m = io.joint ? uint32_t(reinterpret_cast<const uint16_t*>(sslice + R::SLICE_BYTES)[lane])
                         : reinterpret_cast<const uint32_t*>(sslice + R::SLICE_BYTES)[lane];
        if(io.joint) m = moves_of_joint(m);

        uint8_t* rec = sslice + lane * POM_REC_BYTES;
        /* (FREEZE as a run-time mask - an expression of `flags`, or a word of StepIO - cost the kernel 17 % of its speed,
         * 0.127 against 0.109 ms per 1 Mi-env tick, with the same instruction and register counts: the mask must be a
         * compile-time constant per branch of `raw`.  tools/ab keeps the builds of that A/B.) */
        const bool stepped = active && !(rec[R_STATUS] & ((raw ? POM_STATUS_INVALID : (POM_STATUS_DONE | POM_STATUS_INVALID)) |
                                                          (FREEZE ? POM_STATUS_TRUNCATED : 0)));
        warp_tick<TEAMS>(sslice, rec, m, stepped, raw, sslice + R::SLICE_BYTES + 128u,
                         (flags & POM_STEP_CONTINUE_UNDEFINED) ? pomcore::F_INVALID_MASK_CONTINUE : pomcore::F_INVALID_MASK);
        acc.steps += stepped ? 1u : 0u;
        uint32_t st_end = active ? rec[R_STATUS] : 0u;
        if(flags & POM_STEP_AUTORESET)
        {
            const uint32_t st = finish_and_reset(sslice, rec, P, env, active && stepped, true, ep_now, acc);
            if(active && stepped) st_end = st;
        }
        if(status_out && active) status_out[env] = uint8_t(st_end);
        /* after a reset the record is the template's, but tick_rewards reads the agent flags only while the game runs */
        if(REWARDS && active)
            reinterpret_cast<uint32_t*>(io.obs)[env] = pomcore::tick_rewards<TEAMS>(stepped, st_end, *reinterpret_cast<const uint32_t*>(rec + R_AFLAGS));
        if(io.done_bits || io.fin_env)
        {
            /* compact results: which envs ended an episode in this tick, as one bit per env and as a list */
            const bool ended = active && stepped && (st_end & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID)) != 0u;
            const uint32_t em = __ballot_sync(FULL_WARP, ended);
            if(io.done_bits && lane == 0) io.done_bits[s] = em;
            if(io.fin_env && em)
            {
                /* appended to the CTA's list in shared memory (one shared-memory atomic per slice); 148 CTAs x 1 global
                 * atomic per launch instead of one per slice - 11 k atomics on ONE address per tick serialise in the L2
                 * and cost the 0.5 Mi-env step 20 us.  A CTA whose list is full appends to the global list directly. */
                uint32_t* fin = reinterpret_cast<uint32_t*>(smem + R::OFF_FIN);
                const uint32_t k = uint32_t(__popc(em));
                uint32_t pos = 0u;
                if(lane == 0) pos = atomicAdd(fin, k);
                pos = __shfl_sync(FULL_WARP, pos, 0);
                const uint32_t mine = uint32_t(__popc(em & ((1u << lane) - 1u)));
                if(pos + k <= R::FIN_CAP)
                {
                    if(ended)
                    {
                        reinterpret_cast<uint32_t*>(smem + R::OFF_FIN_ENV)[pos + mine] = uint32_t(env);
                        smem[R::OFF_FIN_ST + pos + mine] = uint8_t(st_end);
                    }
                }
                else
                {
                    /* the shared-memory counter only grows: from the first reservation that does not fit, every later
                     * one fails too, so the entries below that position are exactly the ones written (fin[1]) */
                    if(lane == 0) { atomicMin(fin + 1, pos); pos = atomicAdd(io.fin_counter, k); }
                    pos = __shfl_sync(FULL_WARP, pos, 0) + mine;
                    if(ended && pos < io.fin_capacity)
                    {
                        io.fin_env[pos] = uint32_t(env);
                        io.fin_status[pos] = uint8_t(st_end);
                    }
                }
            }
        }
        fence_proxy_async();
        __syncwarp();
        if(lane == 0) bulk_s2g(P.recs + s * R::SLICE_BYTES, sslice, R::SLICE_BYTES);
        if(OBS && io.obs)
        {
            /* what the agents see now: built from the records while they are still in shared memory (the bulk store above
             * only reads them), written straight to HBM - no second pass over the 306 MB record array */
            const uint32_t n_valid = whole ? 32u : uint32_t(P.n_envs - s * 32u);
            uint32_t k = 0u;
            for(int a = 0; a < 4; a++)
            {
                if(!((io.obs_mask >> a) & 1u)) continue;
                warp_observe_slice(sslice, a, io.obs_view, io.obs + (uint64_t(k) * io.obs_stride + s * 32u) * POM_OBS_BYTES, n_valid);
                k++;
            }
        }
        __syncwarp();
        if(lane == 0)
        {
            bulk_wait_read_all();
            __threadfence_block();
            atomicOr(free_mask, 1u << b);                             /* the buffer may be loaded into again */
        }
        __syncwarp();
    }
    acc_flush(P.stats, acc, (flags & POM_STEP_COUNT) != 0u);
    if(io.fin_env)
    {
        /* The last warp of a CTA hands the CTA's list to the global list; the last CTA publishes the length and clears the
         * counters for the next launch (no second kernel).  ONE global round trip per CTA: a 64-bit atomic adds the CTA's
         * entries to the low word (the list position) and 1 to the high word (CTAs done).  No device-wide fences: the
         * caller reads the list after the launch has completed, and the CTA that finds itself last knows the total from
         * the value the atomic returned.  (Reservation, fence, a second atomic for the CTA count and another fence, one
         * after the other at the end of every CTA, cost 3.5 us per launch - tools/e2e_probe.py.) */
        __threadfence_block();
        uint32_t* warps_done = ticket + 1;
        bool last = false;
        if(lane == 0) last = atomicAdd(warps_done, 1u) == uint32_t(NW - 1);
        last = __shfl_sync(FULL_WARP, last ? 1 : 0, 0) != 0;
        if(last)
        {
            __threadfence_block();
            const volatile uint32_t* fin = reinterpret_cast<const volatile uint32_t*>(smem + R::OFF_FIN);
            const uint32_t k = fin[1] != 0xFFFFFFFFu ? fin[1] : fin[0];
            unsigned long long old = 0ull;
            if(lane == 0) old = atomicAdd(reinterpret_cast<unsigned long long*>(io.fin_counter), (1ull << 32) | k);
            old = __shfl_sync(FULL_WARP, old, 0);
            const uint32_t base = uint32_t(old);
            for(uint32_t i = lane; i < k; i += 32u)
            {
                if(base + i < io.fin_capacity)
                {
                    io.fin_env[base + i] = reinterpret_cast<const uint32_t*>(smem + R::OFF_FIN_ENV)[i];
                    io.fin_status[base + i] = smem[R::OFF_FIN_ST + i];
                }
            }
            if(lane == 0 && uint32_t(old >> 32) == gridDim.x - 1u)
            {
                /* every other CTA has made its reservations (also those that went past a full CTA list): base + k is the total */
                const uint32_t count = base + k;
                *io.fin_count_out = count < io.fin_capacity ? count : io.fin_capacity;
                *reinterpret_cast<volatile unsigned long long*>(io.fin_counter) = 0ull;
            }
        }
    }
}

/* ---------------------------------------------------------------- K7: agent memories of the SimpleAgent policy */
/* An env's memories are valid for the episode they were written in: a reset by any path (k_step auto-reset, rollout,
 * pom_batch_reset) bumps or clears episodes[env], and the next reader starts from zeroed agents, which is what four
 * freshly constructed SimpleAgent objects hold (performance_test.cpp:59-61 builds new agents per game). */
struct GlobalAgentStore {
    uint32_t* base;           /* &policy[env] */
    uint64_t  stride;
    __device__ __forceinline__ pompolicy::SimpleSt load(int a) const
    {
        pompolicy::SimpleSt s;
        s.w0 = base[uint64_t(2 * a) * stride];
        s.w1 = base[uint64_t(2 * a + 1) * stride];
        return s;
    }
    __device__ __forceinline__ void store(int a, const pompolicy::SimpleSt& v)
    {
        base[uint64_t(2 * a) * stride] = v.w0;
        base[uint64_t(2 * a + 1) * stride] = v.w1;
    }
    __device__ __forceinline__ void clear(uint32_t episode)
    {
#pragma unroll
        for(int k = 0; k < 8; k++) base[uint64_t(k) * stride] = 0u;
        base[8 * stride] = episode;
    }
    __device__ __forceinline__ void claim(uint32_t episode)
    {
        if(base[8 * stride] != episode) clear(episode);
    }
};

/* FOG (k_policy_moves, k_rollout with POLICY, k_policy_act): the SimpleAgents play under fog of war
 * (pom_batch_set_policy_view, pompolicy::simple_moves).  The view, 0..15, is a run-time value that travels in spare bits
 * of an existing argument: bits POLICY_VIEW_SHIFT.. of the agent mask, of k_policy_act's draw.  (A view of 15 sees every
 * position a record can hold, so larger views are passed as 15.) */
constexpr uint32_t POLICY_VIEW_SHIFT = 8;

/* per-tick mode: moves[env] byte a <- SimpleAgent::act for every agent a in `mask` of every running env (IDLE for a dead
 * agent); the other bytes are kept.  Records are staged read-only with the same per-warp bulk load as k_step. */
template<int TPB, bool TEAMS = false, bool FOG = false>
__global__ void __launch_bounds__(TPB) k_policy_moves(BatchParams P, uint32_t* __restrict__ moves, uint64_t seed, uint32_t tick, uint32_t mask,
                                                     uint32_t gen_actions, uint32_t freeze_truncated)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const uint64_t env = uint64_t(blockIdx.x) * TPB + threadIdx.x;
    const bool active = env < P.n_envs;
    constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + TileScratch<TPB>::OFF_BAR) + warp;
    uint8_t* sslice = smem + warp * SLICE_BYTES;
    const uint8_t* gslice = P.recs + (size_t(blockIdx.x) * TPB + warp * 32u) * POM_REC_BYTES;
    if(lane == 0)
    {
        mbar_init(bar, 1);
        fence_barrier_init();
        mbar_expect_tx(bar, SLICE_BYTES);
        bulk_g2s(sslice, gslice, SLICE_BYTES, bar);
    }
    /* gen_actions != 0: the agents outside the mask play uniform random moves from the shared counter RNG (what the fused
     * rollout does); else their bytes are the caller's */
    uint32_t m = !active ? 0u : (gen_actions ? pomcore::rng_moves(seed, P.env_offset + env, tick, gen_actions) : moves[env]);
    const uint32_t ep = active ? P.episodes[env] : 0u;
    const uint32_t draws = pomcore::rng_moves(seed, P.env_offset + env, tick, 5u);
    __syncwarp();
    mbar_wait(bar, 0);
    const uint8_t* rec = sslice + lane * POM_REC_BYTES;
    if(active && !(rec[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID | (freeze_truncated ? POM_STATUS_TRUNCATED : 0u))))
    {
        GlobalAgentStore S{ P.policy + env, P.policy_stride };
        S.claim(ep);
        if constexpr(FOG) m = pompolicy::simple_moves<TEAMS, true>(rec, mask, m, draws, S, int(mask >> POLICY_VIEW_SHIFT));
        else m = pompolicy::simple_moves<TEAMS>(rec, mask, m, draws, S);
        moves[env] = m;
    }
    else if(active && gen_actions) moves[env] = m;
}

/* ---------------------------------------------------------------- K2: fused K-tick rollout */
/* POLICY = false: uniform random agents only (the headline rollout; no policy code in the kernel image).
 * POLICY = true : the agents in `policy_mask` play SimpleAgent, the others stay uniform random. */
/* SPEC: the image of the headline rollout (uniform{0..5} agents from the counter RNG, auto-reset, default handling of
 * the undefined states) with those choices known at compile time */
template<int TPB, bool POLICY, bool SPEC = false, bool TEAMS = false, bool FOG = false>
__global__ void __launch_bounds__(TPB) k_rollout(BatchParams P, uint32_t ticks, uint64_t seed, uint32_t tick0,
                                                uint32_t n_actions_in, uint32_t roll_flags_in, uint32_t policy_mask,
                                                const uint32_t* __restrict__ move_seq_in)
{
    const uint32_t n_actions = SPEC ? 6u : n_actions_in, roll_flags = SPEC ? 0u : roll_flags_in;
    const uint32_t* __restrict__ move_seq = SPEC ? nullptr : move_seq_in;
    const uint32_t no_reset = (roll_flags & POM_ROLL_NO_RESET) ? 1u : 0u;
    const int invalid_mask = (roll_flags & POM_ROLL_CONTINUE_UNDEFINED) ? pomcore::F_INVALID_MASK_CONTINUE : pomcore::F_INVALID_MASK;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint64_t env = uint64_t(blockIdx.x) * TPB + threadIdx.x;
    const bool active = env < P.n_envs;
    constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + TileScratch<TPB>::OFF_BAR) + warp;
    uint8_t* sslice = smem + warp * SLICE_BYTES;
    uint8_t* gslice = P.recs + (size_t(blockIdx.x) * TPB + warp * 32u) * POM_REC_BYTES;
    if(lane == 0)
    {
        mbar_init(bar, 1);
        fence_barrier_init();
        mbar_expect_tx(bar, SLICE_BYTES);
        bulk_g2s(sslice, gslice, SLICE_BYTES, bar);
    }
    uint32_t ep_now = active ? P.episodes[env] : 0u;
    /* agent memories stay in global memory (word-major, so every access of a warp is one coalesced 128-byte line that
     * lives in L1/L2 for the whole rollout): keeping them in shared memory would cost one resident CTA per SM */
    GlobalAgentStore agents{ P.policy + (active ? env : 0), P.policy_stride };
    if(POLICY && active) agents.claim(ep_now);
    __syncwarp();
    mbar_wait(bar, 0);

    uint8_t* rec = sslice + lane * POM_REC_BYTES;
    /* per-env RNG key hoisted out of the tick loop (first splitmix64 of pom_rng_moves) */
    const uint64_t key = pomcore::splitmix64(seed ^ ((P.env_offset + env) * 0xD6E8FEB86659FD93ull));
    EpisodeAcc acc;
    for(uint32_t k = 0; k < ticks; k++)
    {
        if((k & 0x3FFFu) == 0x3FFFu) acc_flush(P.stats, acc, true);   /* the per-lane counters are 16 bits wide */
        const bool stepped = active && !(rec[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID));
        uint32_t m = 0;
        if(stepped && move_seq)
        {
            /* pom_batch_step_seq: the caller's moves, tick-major; one coalesced 4-byte load per env and tick */
            m = __ldg(move_seq + uint64_t(k) * P.n_envs + env);
            acc.steps++;
        }
        else if(stepped)
        {
            const uint64_t h = pomcore::splitmix64(key + uint64_t(tick0 + k));
#pragma unroll
            for(int a = 0; a < 4; a++)
                m |= (((uint32_t(h >> (16 * a)) & 0xFFFFu) * n_actions) >> 16) << (8 * a);
            if(POLICY)
            {
                uint32_t draws = 0;
#pragma unroll
                for(int a = 0; a < 4; a++)
                    draws |= (((uint32_t(h >> (16 * a)) & 0xFFFFu) * 5u) >> 16) << (8 * a);
                if constexpr(FOG) m = pompolicy::simple_moves<TEAMS, true>(rec, policy_mask, m, draws, agents, int(policy_mask >> POLICY_VIEW_SHIFT));
                else m = pompolicy::simple_moves<TEAMS>(rec, policy_mask, m, draws, agents);
            }
            acc.steps++;
        }
        warp_tick<TEAMS>(sslice, rec, m, stepped, false, smem + TileScratch<TPB>::OFF_LIST + 8u * warp, invalid_mask);
        const uint32_t st = finish_and_reset(sslice, rec, P, env, active && stepped, !no_reset, ep_now, acc);
        /* a new episode starts with four new agents */
        if(POLICY && stepped && !no_reset && (st & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID))) agents.clear(ep_now);
    }
    acc_flush(P.stats, acc, true);

    fence_proxy_async();
    __syncwarp();
    if(lane == 0)
    {
        bulk_s2g(gslice, sslice, SLICE_BYTES);
        bulk_wait_read_all();
    }
}

/* SimpleAgent::act for ONE agent of ONE env with a caller-chosen draw (the host mirror's agents::SimpleAgent) */
template<bool TEAMS = false, bool FOG = false>
__global__ void k_policy_act(BatchParams P, uint64_t env, int agent, uint32_t draw, int* move_out)
{
    const uint8_t* rec = P.recs + env * POM_REC_BYTES;
    GlobalAgentStore S{ P.policy + env, P.policy_stride };
    S.claim(P.episodes[env]);
    const pompolicy::Boards B = pompolicy::make_boards(rec);
    pompolicy::SimpleSt st = S.load(agent);
    if constexpr(FOG) *move_out = int(pompolicy::simple_act<TEAMS, true>(rec, B, agent, st, draw & 0xFFu, int(draw >> POLICY_VIEW_SHIFT)));
    else *move_out = int(pompolicy::simple_act<TEAMS>(rec, B, agent, st, draw));
    S.store(agent, st);
}

/* agent memories <-> array of pom_simple_agent[4] per env (8 words), applying the episode rule */
__global__ void k_policy_export(BatchParams P, uint64_t first, uint64_t count, uint32_t* __restrict__ out)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i >= count) return;
    const uint64_t env = first + i;
    const bool mine = P.policy[8 * P.policy_stride + env] == P.episodes[env];
    for(int k = 0; k < 8; k++) out[8 * i + k] = mine ? P.policy[uint64_t(k) * P.policy_stride + env] : 0u;
}

__global__ void k_policy_import(BatchParams P, uint64_t first, uint64_t count, const uint32_t* __restrict__ in)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i >= count) return;
    const uint64_t env = first + i;
    for(int k = 0; k < 8; k++) P.policy[uint64_t(k) * P.policy_stride + env] = in[8 * i + k];
    P.policy[8 * P.policy_stride + env] = P.episodes[env];
}

/* ---------------------------------------------------------------- K3: templates and (re)initialisation */
/* one thread per candidate seed; the 2.5 KB Mersenne state lives in local memory (init is off the hot path) */
__global__ void k_make_templates(uint8_t* out_recs, uint8_t* dirty, int first_seed, uint32_t n_candidates)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if(i >= n_candidates) return;
    pomcore::Mt64 g;
    uint8_t rec[POM_REC_BYTES];
    const int d = pomcore::init_record(rec, g, first_seed + int(i), 0, 1, 2, 3);
    dirty[i] = uint8_t(d);
    uint8_t* o = out_recs + size_t(i) * POM_REC_BYTES;
    for(int k = 0; k < POM_REC_BYTES; k++) o[k] = rec[k];
}

/* compaction of the clean candidates into the pool: pool[k] <- cand[pick[k]] (word copy) */
__global__ void k_gather_records(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src,
                                 const uint32_t* __restrict__ idx, uint64_t n_dst, uint64_t dst_first)
{
    const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(t >= n_dst * POM_REC_WORDS) return;
    const uint64_t e = t / POM_REC_WORDS;
    const uint32_t w = uint32_t(t - e * POM_REC_WORDS);
    dst[(dst_first + e) * POM_REC_WORDS + w] = __ldg(src + uint64_t(idx[e]) * POM_REC_WORDS + w);
}

/* env e <- template[(env_offset + e + episode[e]) % n_templates]; episode numbers as given */
__global__ void k_fill_from_templates(BatchParams P)
{
    const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(t >= P.n_envs * POM_REC_WORDS) return;
    const uint64_t e = t / POM_REC_WORDS;
    const uint32_t w = uint32_t(t - e * POM_REC_WORDS);
    const uint64_t k = (P.env_offset + e + P.episodes[e]) % P.n_templates;
    reinterpret_cast<uint32_t*>(P.recs)[t] = __ldg(reinterpret_cast<const uint32_t*>(P.templates) + k * POM_REC_WORDS + w);
}

/* ---------------------------------------------------------------- K4: tree-search expansion */
/* child c = root_i * fanout + j: copy the root's record into the tile, apply joint action j
 * (a_k = (j / 6^k) % 6), Step once, bulk-store the tile.
 * The tile is filled by the whole warp: the 32 children of a slice share one root (two where a slice straddles a root
 * boundary; fanout >= 32 in a tree search), so the lanes fetch the root's 73 words ONCE with three coalesced loads and
 * replicate them from registers into the 32 records - 96 conflict-free shared-memory stores per lane, no load between
 * them.  (The first form had every lane copy its own record word by word: 73 dependent load -> store pairs per lane,
 * one in flight at a time, 0.55 of the HBM write peak.) */
template<int TPB, bool TEAMS = false>
__global__ void __launch_bounds__(TPB) k_expand_step(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src,
                                                    const uint32_t* __restrict__ src_idx, uint64_t n_children,
                                                    uint32_t fanout, uint32_t flags)
{
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint64_t c0 = uint64_t(blockIdx.x) * TPB + warp * 32u;      /* first child of this warp's slice */
    if(c0 >= n_children) return;
    const uint64_t c = c0 + lane;
    uint8_t* sslice = smem + warp * SLICE_BYTES;
    uint8_t* rec = sslice + lane * POM_REC_BYTES;
    uint32_t* sw = reinterpret_cast<uint32_t*>(sslice);
    const bool raw = (flags & POM_STEP_RAW) != 0u;

    const uint64_t root0 = c0 / fanout;
    const uint32_t j0 = uint32_t(c0 - root0 * fanout);
    const uint32_t n_here = uint32_t(n_children - c0 < 32u ? n_children - c0 : 32u);
    {
        uint64_t root = root0;
        uint32_t j = j0, w0 = 0u, w1 = 0u, w2 = 0u;
        bool have = false;
#pragma unroll 4
        for(uint32_t r = 0; r < 32u; r++)
        {
            if(r >= n_here) { w0 = w1 = w2 = 0u; have = true; }       /* lanes behind the last child hold empty records */
            else if(!have)
            {
                const uint32_t* s = reinterpret_cast<const uint32_t*>(src + size_t(__ldg(src_idx + root)) * POM_REC_BYTES);
                w0 = __ldg(s + lane);
                w1 = __ldg(s + lane + 32u);
                w2 = lane < uint32_t(POM_REC_WORDS - 64) ? __ldg(s + lane + 64u) : 0u;
                have = true;
            }
            uint32_t* d = sw + r * POM_REC_WORDS;
            d[lane] = w0;
            d[lane + 32u] = w1;
            if(lane < uint32_t(POM_REC_WORDS - 64)) d[lane + 64u] = w2;
            if(++j == fanout) { j = 0u; root++; have = false; }      /* warp-uniform */
        }
    }
    __syncwarp();
    uint32_t m = 0u;
    bool stepped = false;
    if(c < n_children)
    {
        uint32_t j = j0 + lane;
        while(j >= fanout) j -= fanout;                               /* fanout may be smaller than 32 */
        m = moves_of_joint(j);
        stepped = !(rec[R_STATUS] & (raw ? POM_STATUS_INVALID : (POM_STATUS_DONE | POM_STATUS_INVALID)));
    }
    warp_tick<TEAMS>(sslice, rec, m, stepped, raw, smem + TileScratch<TPB>::OFF_LIST + 8u * warp,
                     (flags & POM_STEP_CONTINUE_UNDEFINED) ? pomcore::F_INVALID_MASK_CONTINUE : pomcore::F_INVALID_MASK);
    if(n_here == 32u)
    {
        fence_proxy_async();
        __syncwarp();
        if(lane == 0)
        {
            bulk_s2g(dst + c0 * POM_REC_BYTES, sslice, SLICE_BYTES);
            bulk_wait_read_all();
        }
    }
    else
    {
        /* the last, partly filled slice: only the children's own records are written - dst envs behind n_children keep
         * their contents (a bulk store of the whole slice would overwrite up to 31 of them) */
        __syncwarp();
        uint32_t* out = reinterpret_cast<uint32_t*>(dst + c0 * POM_REC_BYTES);
        for(uint32_t w = lane; w < n_here * uint32_t(POM_REC_WORDS); w += 32u) out[w] = sw[w];
    }
}

/* ---------------------------------------------------------------- K5: AoS <-> packed */
__global__ void k_pack(const pom_state* __restrict__ aos, const uint8_t* __restrict__ status, uint8_t* recs,
                       uint64_t first, uint64_t count, uint32_t* bad_count)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i >= count) return;
    const int bad = pomcore::pack(aos + i, status ? status[i] : uint8_t(0), recs + (first + i) * POM_REC_BYTES);
    if(bad) atomicAdd(bad_count, 1u);
}

__global__ void k_unpack(const uint8_t* __restrict__ recs, pom_state* aos, uint8_t* status, uint64_t first, uint64_t count)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i >= count) return;
    if(aos)
    {
        const uint8_t st = pomcore::unpack(recs + (first + i) * POM_REC_BYTES, aos + i);
        if(status) status[i] = st;
    }
    else if(status) status[i] = recs[(first + i) * POM_REC_BYTES + R_STATUS];
}

/* the State of env first + i as agent `agent` sees it through a window of `view` cells (pomcore::fog_state) */
__global__ void k_observe(const uint8_t* __restrict__ recs, pom_state* aos, uint8_t* status, uint64_t first, uint64_t count, int agent, int view)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i >= count) return;
    const uint8_t st = pomcore::unpack(recs + (first + i) * POM_REC_BYTES, aos + i);
    pomcore::fog_state(aos + i, agent, view);
    if(status) status[i] = st;
}

/* observation planes for the agents in `mask`, written as POM_OBS_BYTES records into one slab per agent:
 * out[((k * stride) + env) * POM_OBS_BYTES], k = rank of the agent within the mask.  Same per-warp staging as k_step: the
 * warp's 32 records come in with one bulk load; the quads of the warp then write the observations straight to the slab
 * (warp_observe_slice).  History: round 1 staged the 32 x 496 bytes in shared memory and bulk-stored them (25 KB per
 * warp, 8 warps per SM, 0.53 of the HBM peak); one lane per env with 32-byte stores needs no tile but makes every
 * lane's store a line of its own (L1 data pipe 67 % busy, 0.164 ms per 1 Mi envs on the bench's states); four lanes
 * per env store whole lines.  The fused form is StepIO::obs. */
/* CROPPED: the image for the cropped layout (with both layouts in one image the kernel needed 127 registers and the full
 * layout lost a third of its speed) */
template<int TPB, bool CROPPED = false>
__global__ void __launch_bounds__(TPB, CROPPED ? 768 / TPB : 0) k_observe_planes(BatchParams P, uint8_t* __restrict__ out, uint64_t stride, uint32_t mask, int view,
                                                                  uint32_t reverse, uint32_t cropped_bytes)
{
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr uint32_t SLICE_BYTES = 32 * POM_REC_BYTES;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    /* `reverse`: the tiles are taken from the end of the batch - right after a step that walked forwards, its last
     * records are still in L2 */
    const uint64_t tile = reverse ? gridDim.x - 1u - blockIdx.x : blockIdx.x;
    const uint64_t env0 = tile * TPB + warp * 32u;                              /* first env of this warp's slice */
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + TileScratch<TPB>::OFF_BAR) + warp;
    uint8_t* sslice = smem + warp * SLICE_BYTES;
    if(lane == 0)
    {
        mbar_init(bar, 1);
        fence_barrier_init();
        mbar_expect_tx(bar, SLICE_BYTES);
        bulk_g2s(sslice, P.recs + env0 * POM_REC_BYTES, SLICE_BYTES, bar);
    }
    __syncwarp();
    mbar_wait(bar, 0);
    if(env0 >= P.n_envs) return;
    const uint32_t n_valid = P.n_envs - env0 < 32u ? uint32_t(P.n_envs - env0) : 32u;
    uint32_t k = 0;
    for(int a = 0; a < 4; a++)
    {
        if(!((mask >> a) & 1u)) continue;
        if(CROPPED) warp_observe_slice_cropped(sslice, a, view, out + (uint64_t(k) * stride + env0) * cropped_bytes, n_valid, cropped_bytes);
        else warp_observe_slice(sslice, a, view, out + (uint64_t(k) * stride + env0) * POM_OBS_BYTES, n_valid);
        k++;
    }
}

/* ---------------------------------------------------------------- misc */
__global__ void k_generate_moves(uint32_t* moves, uint64_t n, uint64_t env_offset, uint64_t seed, uint32_t tick, uint32_t n_actions)
{
    const uint64_t e = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(e < n) moves[e] = pomcore::rng_moves(seed, env_offset + e, tick, n_actions);
}

__global__ void k_apply(uint8_t* recs, uint64_t env, int op, int a0, int a1, int a2)
{
    uint8_t* rec = recs + env * POM_REC_BYTES;
    pomcore::Agents A;
    pomcore::load_agents(rec, A);
    int flags = 0;
    if(op == POM_OP_SPAWN_FLAME) pomcore::explode(rec, A, uint32_t(a0) | (uint32_t(a1) << 4), uint32_t(a2), 31u, flags);
    else if(op == POM_OP_EXPLODE_TOP && rec[R_BCOUNT] > 0)
    {
        const uint32_t c = pomcore::bomb_at(rec, 0);
        pomcore::explode(rec, A, c & 0xFFu, (c >> 12) & 15u, 31u, flags);
        const int id = int((pomcore::bomb_at(rec, 0) >> 8) & 3u);
        A.bcnt = pomcore::with_byte(A.bcnt, id, pomcore::byte_of(A.bcnt, id) - 1u);
        rec[R_BINDEX] = uint8_t(pomcore::ring_next(rec[R_BINDEX]));
        rec[R_BCOUNT] = uint8_t(rec[R_BCOUNT] - 1);
    }
    else if(op == POM_OP_EXPLODE_AT && a0 >= 0 && a0 < int(rec[R_BCOUNT]))
    {
        const uint32_t eb = pomcore::bomb_at(rec, a0);
        pomcore::explode(rec, A, eb & 0xFFu, pomcore::byte_of(A.astr, int((eb >> 8) & 3u)), uint32_t(a0), flags);
    }
    else if(op == POM_OP_POP_FLAME && rec[R_FCOUNT] > 0) pomcore::pop_flame(rec);
    pomcore::store_agents(rec, A);
    if(flags & pomcore::F_INVALID_MASK) rec[R_STATUS] |= POM_STATUS_INVALID;
}

/* one seed -> zero-initialised State + InitBoardItems (no agents placed) */
__global__ void k_make_board(uint8_t* out_rec, uint8_t* dirty, int seed)
{
    pomcore::Mt64 g;
    uint8_t rec[POM_REC_BYTES];
    dirty[0] = uint8_t(pomcore::init_board(rec, g, seed));
    for(int k = 0; k < POM_REC_BYTES; k++) out_rec[k] = rec[k];
}

__global__ void k_fill_zero(uint4* p, uint64_t n16)
{
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if(i < n16) p[i] = make_uint4(0u, 0u, 0u, 0u);
}

}

#endif
