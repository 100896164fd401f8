/*
 * pom_batch.h — C ABI of the B200-native batched Pommerman step path (libpom_b200.so).
 *
 * The reference (dist1ll/pomcpp) has no FFI layer: consumers include include/bboard.hpp and link
 * lib/pomlib.a (README.md:58-60, Makefile:34-38).  These entry points are what a binding of the
 * step path replaces; each one cites the reference interface it stands for.  All states live on
 * ONE GPU per handle as packed 292-byte records (pomcpp_b200/csrc/pom_record.h); host buffers use
 * the AoS `pom_state` of pom_state.h, which is layout-identical to the reference's bboard::State.
 *
 * Conventions
 *   - every function returns 0 on success or a negative POM_E_* code; nothing throws across the ABI;
 *     pom_last_error() returns a thread-local description of the last failure.
 *   - a handle owns its device buffers and one CUDA stream; calls on one handle are stream-ordered
 *     and NOT thread-safe; different handles (e.g. one per GPU) may be driven from different threads.
 *   - functions taking host pointers synchronise before returning; pom_batch_step / _rollout /
 *     _clone / _expand_step only enqueue work (use pom_batch_sync, or CUDA events on pom_batch_stream).
 *   - there is no CPU fallback: without a CUDA device pom_batch_init fails with POM_E_CUDA.
 */
#ifndef POM_BATCH_H_
#define POM_BATCH_H_

#include <stdint.h>
#include "pom_state.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pom_batch pom_batch;

enum {
    POM_OK        =  0,
    POM_E_ARG     = -1,   /* bad argument                                   */
    POM_E_CUDA    = -2,   /* CUDA runtime error (see pom_last_error)         */
    POM_E_NOMEM   = -3,   /* device or host allocation failed                */
    POM_E_RANGE   = -4,   /* env index / count outside the batch             */
    POM_E_STATE   = -5    /* an uploaded state cannot be represented (envs marked POM_STATUS_INVALID) */
};

/* flags of pom_batch_step / pom_batch_expand_step */
enum {
    POM_STEP_RAW       = 0x1, /* bare bboard::Step (step.cpp:9): no timeStep++, no done/winner, finished envs are stepped too */
    POM_STEP_AUTORESET = 0x2, /* an env that finishes IN THIS TICK is counted in the stats and re-initialised from the
                                 template pool at the end of the tick (not in the reference).  An env that is already
                                 done or invalid when the tick starts (uploaded that way, or finished by an earlier
                                 step without this flag) is not stepped and therefore stays frozen: use pom_batch_reset,
                                 or upload a running state */
    POM_STEP_COUNT     = 0x4, /* add the number of envs stepped to stats.env_steps                       */
    POM_STEP_CONTINUE_UNDEFINED = 0x10, /* Where the reference dereferences a null bomb (step.cpp:167, a kicker walks onto a
                                 BOMB cell without queue entry) or recurses without end (step_utility.cpp:89-92, the
                                 reversion chain reaches an agent that did not move), the env is by default marked
                                 POM_STATUS_INVALID and frozen (counted in stats.invalid).  With this flag it keeps
                                 running with the canonical result instead: the kicker moves and no bomb gets a
                                 direction; the chain stops at that agent.  Queue overflows and values the record cannot
                                 carry still invalidate.  The reference has no behaviour to compare with here. */
    POM_STEP_OVERLAP   = 0x8  /* pom_batch_step only: step the two halves of the batch on two internal streams so that
                                 consecutive ticks overlap at their edges.  Every other call on the handle first waits
                                 for both halves; work the caller enqueues DIRECTLY on pom_batch_stream() is ordered after
                                 the first half only - call pom_batch_sync or any other entry point first. */
};

/* flags of pom_batch_rollout: actions per agent come from the shared stateless RNG
 * (see pom_rng_moves); POM_ROLL_HARMLESS draws from {0..4} (HarmlessAgent, basic_agents.cpp:28-38),
 * default is {0..5} (RandomAgent, basic_agents.cpp:12-22). */
enum {
    POM_ROLL_HARMLESS  = 0x1,
    POM_ROLL_NO_RESET  = 0x2, /* finished envs freeze (Environment::Step, environment.cpp:125-128) instead of auto-resetting */
    POM_ROLL_CONTINUE_UNDEFINED = 0x4, /* as POM_STEP_CONTINUE_UNDEFINED */
    /* bits 8..11: agent a plays the reference's heuristic SimpleAgent (simple_agent.cpp:12-141) instead of drawing
     * uniformly; the reference's own benchmark runs four of them (performance_test.cpp:38,59-63) */
    POM_ROLL_SIMPLE_SHIFT = 8
};
#define POM_ROLL_SIMPLE(agent_mask) (((uint32_t)(agent_mask) & 0xFu) << POM_ROLL_SIMPLE_SHIFT)

/* How pom_batch_init fills the batch.  Replaces InitState / InitBoardItems / PutAgentsInCorners
 * (bboard.hpp:651,661; bboard.cpp:322-382) and Environment::MakeGame (environment.cpp:53-66). */
typedef struct pom_init_desc {
    uint64_t         env_offset;      /* global index of this handle's env 0 (sharding over GPUs)            */
    uint32_t         n_templates;     /* size of the template pool kept on the device (>= 1)                 */
    int32_t          first_seed;      /* pool = InitState(s, 0,1,2,3) for the first n_templates seeds >= first_seed that
                                         are free of the reference's uninitialised-read defect (bboard.cpp:351,367,372),
                                         generated ON THE DEVICE (mt19937_64 + libstdc++ uniform_int_distribution)   */
    const pom_state* host_templates;  /* if non-NULL: n_templates AoS states to use as the pool instead             */
    uint32_t         max_ticks;       /* rollout truncation (Pommerman: 800); 0 = never.  timeStep is 16 bits on the
                                         device, so values above 65535 never truncate: an env that plays on is aborted
                                         as POM_STATUS_INVALID on its 65 536th tick instead (timeStep stays 65535) */
    uint32_t         flags;           /* POM_INIT_*                                                            */
} pom_init_desc;

enum {
    POM_INIT_EMPTY = 0x1,  /* do not fill the envs (they will be uploaded); the pool is still built */
    POM_INIT_TEAMS = 0x2,  /* the handle plays the 2v2 TEAM game: team 0 = agents 0 and 2, team 1 = agents 1 and 3.
                              Step (bboard::Step) is the same, flames kill teammates too; what changes is when an episode
                              ends and who won (pom_state.h: the status byte) and whom the device SimpleAgent treats as an
                              enemy (not its teammate).  The reference has no team mode: this is the project's definition.
                              The mode is fixed for the handle's life and applies to every entry point that steps or acts;
                              pom_batch_clone / pom_batch_expand_step between handles of different modes fail (POM_E_ARG). */
    POM_INIT_RADIO = 0x4   /* the team game with the TEAM RADIO of Pommerman's team-radio environment (pommerman/envs/v2.py, the
                              NeurIPS 2018 competition format): every tick each agent sends its teammate two words of 0..7,
                              which the teammate reads in its next observation (pom_batch_step_radio).  Needs POM_INIT_TEAMS
                              (POM_E_ARG otherwise); fixed for the handle's life.  pom_batch_clone / pom_batch_expand_step
                              between a radio and a non-radio handle fail (POM_E_ARG). */
};

/* episode counters accumulated on the device (Environment::IsDone/IsDraw/GetWinner, bboard.hpp:617-631) */
typedef struct pom_stats {
    uint64_t env_steps;        /* Steps executed (finished/frozen envs not counted) */
    uint64_t episodes;         /* episodes finished (won + draw + truncated + invalid) */
    uint64_t wins[4];          /* episodes won by agent 0..3; team game: wins[t] by team t, wins[2] = wins[3] = 0 */
    uint64_t draws;            /* aliveAgents == 0; team game: both teams out in the same tick */
    uint64_t truncated;        /* timeStep reached max_ticks                         */
    uint64_t sum_episode_len;  /* sum of timeStep over finished episodes             */
    uint64_t invalid;          /* episodes aborted because the env left the reference's defined domain
                                  (the reference itself would crash or hang there, SURVEY §8c D3-D5), or
                                  because it reached the 16-bit timeStep ceiling (see max_ticks).  An episode that
                                  ends DONE or TRUNCATED in that same tick counts there, not here */
} pom_stats;
#define POM_STATS_WORDS 10

/* ---- lifetime ---- */
int  pom_device_count(void);
int  pom_batch_init(pom_batch** out, int device, uint64_t n_envs, const pom_init_desc* desc);
int  pom_batch_destroy(pom_batch* b);
int  pom_batch_sync(pom_batch* b);
const char* pom_last_error(void);
/* 1 if the handle plays the team game (POM_INIT_TEAMS), 0 for free-for-all, POM_E_ARG for a null handle */
int  pom_batch_teams(const pom_batch* b);
/* 1 if the handle has the team radio (POM_INIT_RADIO), 0 if not, POM_E_ARG for a null handle */
int  pom_batch_radio(const pom_batch* b);
/* *out = 1 if the handle's record array lives in compressible device memory (granted by the driver where the device
 * supports generic compression; the array is then rounded up to the allocation granularity), 0 if it came from
 * cudaMalloc.  A read-only report of what the handle got: results are the same either way. */
int  pom_batch_records_compressed(const pom_batch* b, int* out);

/* ---- AoS <-> packed exchange (there is no reference call: State is passed by pointer) ---- */
int  pom_batch_upload(pom_batch* b, uint64_t first, uint64_t count, const pom_state* states, const uint8_t* status /* may be NULL */);
int  pom_batch_download(pom_batch* b, uint64_t first, uint64_t count, pom_state* states /* may be NULL */, uint8_t* status /* may be NULL */);
/* like pom_batch_download, but every State is what agent `agent` observes through a square window of `view` cells
 * around its position (Pommerman: 4): cells outside are Item::FOG (bboard.hpp:62), agents / bombs / flames outside are
 * not exposed (bboard.hpp:218-226: "if someone is out of sight we simply don't expose their AgentInfo"; hidden agents
 * keep only `dead`, x = y = -1).  The reference declares this ("potentially fogged board state", bboard.hpp:529) but
 * never implements it.  The result is what Agent::act(const State*) is meant to receive. */
int  pom_batch_observe(pom_batch* b, uint64_t first, uint64_t count, int agent, int view, pom_state* states, uint8_t* status);
/* The same view as byte planes for a network input, written on the device (nothing crosses PCIe).
 * One observation = POM_OBS_BYTES (512) bytes, 496 of content and 16 of zero padding, so that every record is 32-byte
 * aligned and a thread can write it with sixteen 256-bit stores (full 32-byte sectors):
 *     0..120   board: the game's item ids in the reference's Item order (bboard.hpp:54-71): 0 passage, 1 rigid, 2 wood,
 *              3 bomb, 4 flames, 5 fog, 6 extra bomb, 7 incr range, 8 kick, 9 agent dummy, 10 + i agent i; index x + 11*y;
 *              powerups hidden in wood / carried by flames are not shown
 *   121..241   blast strength of the visible bomb whose queue entry sits on the cell (0 = none)
 *   242..362   its timer (1..10)
 *   363..483   ticks the visible flame on the cell still burns (timeLeft of its flame-queue entry)
 *   484 x  485 y  486 ammo = maxBombCount - bombCount (clamped to 0..255)  487 blast strength  488 can kick
 *   489 alive mask (bit i = agent i alive; public)  490..491 timeStep (little endian)  492 observer alive  493..511 zero
 *   (on a radio handle, POM_INIT_RADIO: 493 = w0 and 494 = w1 of the teammate's last message, pom_batch_step_radio)
 * Cells outside the window hold 5 (fog) in the board plane and 0 elsewhere.
 * obs_dev: DEVICE buffer of popcount(agent_mask) slabs of pom_batch_obs_stride(b) observations each; the observation of
 * env e for the k-th agent of the mask (in agent order) starts at ((k * stride) + e) * POM_OBS_BYTES.  The stride is
 * n_envs rounded up to a multiple of 256; the tail of each slab is scratch. */
#define POM_OBS_BYTES 512
uint64_t pom_batch_obs_stride(const pom_batch* b);
int  pom_batch_observe_planes(pom_batch* b, uint8_t* obs_dev, uint32_t agent_mask, int view);
/* The CROPPED layout of the same observation: only the window.  With W = 2 * view + 1 (view 0..5) one observation is
 * pom_obs_cropped_bytes(view) = 4 * W * W + 12 bytes rounded up to a multiple of 32 (view 4: 352 instead of 512):
 *     p * W * W + row * W + col   plane p (0 board ids, 1 blast strength, 2 bomb timer, 3 flame life, as above) of board
 *                                 cell (x - view + col, y - view + row), (x, y) = the observer's position; window cells
 *                                 that lie off the board hold 5 (fog) in the board plane and 0 elsewhere
 *     4 * W * W ... + 11          the twelve scalar bytes 484..495 of the full layout, then zero padding (so on a radio
 *                                 handle the teammate's message is in bytes 4 W W + 9 and 4 W W + 10)
 * Slabs as for pom_batch_observe_planes, with pom_obs_cropped_bytes(view) in place of POM_OBS_BYTES. */
uint32_t pom_obs_cropped_bytes(int view);   /* 0 for a view outside 0..5 */
int  pom_batch_observe_planes_cropped(pom_batch* b, uint8_t* obs_dev, uint32_t agent_mask, int view);
int  pom_batch_reset(pom_batch* b);   /* all envs back to their template, counters and episode numbers cleared */
int  pom_batch_templates(pom_batch* b, pom_state* out /* n_templates */, int32_t* seeds_out /* may be NULL */);

/* ---- the hot path ---- */
/* bboard::Step(State*, Move*) (bboard.hpp:668, step.cpp:9-284) wrapped in Environment::Step's
 * bookkeeping (environment.cpp:125-128,149-168) for every env.  moves_dev: DEVICE pointer to
 * n_envs x 4 bytes, byte a of env e = Move of agent a (bboard.hpp:35-43), values 0..5.         */
int  pom_batch_step(pom_batch* b, const uint8_t* moves_dev, uint32_t flags);
/* same with HOST buffers: copies moves in, steps, copies the status bytes out (may be NULL), synchronises.
 * status_host[e] is the env's status at the END of this tick; with POM_STEP_AUTORESET it is the status of the
 * episode that just ended (done / winner / draw / truncated / invalid) even though the env itself has already
 * been re-initialised — the "done" signal an RL loop needs.
 * Buffers from pom_host_alloc (or any page-locked, device-mapped memory) are read and written by the kernel directly
 * over PCIe; pageable buffers are staged through chunked asynchronous copies.                             */
int  pom_batch_step_host(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags);
/* the same without the final synchronisation, for page-locked mapped buffers only (pom_host_alloc): returns as soon as
 * the step is queued; status_host (and moves_host) belong to the device until pom_batch_sync(b) returns.  Lets a caller
 * that runs two batches alternately keep the GPU busy while it consumes the results of the other batch. */
int  pom_batch_step_host_async(pom_batch* b, const uint8_t* moves_host, uint8_t* status_host, uint32_t flags);
/* One tick with COMPACT input and output, for actor loops whose bottleneck is the host link (PCIe / host memory), e.g.
 * eight GPUs fed from one host: 2 bytes in and ~0.3 bytes out per env-step instead of 4 + 1.
 *   joint      n_envs joint actions, j = a0 + 6*a1 + 36*a2 + 216*a3 with a_k = Move of agent k (the encoding of
 *              pom_batch_expand_step).  All four moves are always supplied, as the reference's Step reads them all
 *              (step_utility.cpp:138-144).  j >= 1296 is taken modulo 6 per digit.
 *   done_bits  (n_envs + 31) / 32 words: bit (e % 32) of word e / 32 = env e ended an episode in this tick
 *              (done, truncated or invalid; with POM_STEP_AUTORESET the env has already been re-initialised).  May be NULL.
 *   fin_env, fin_status, fin_count   the same envs as a compacted list in no particular order: env index and status byte
 *              (as pom_batch_step_host's status_host reports it), *fin_count entries, at most fin_capacity (further
 *              ones are dropped: size the list for the worst case n_envs, or poll done_bits).  fin_env may be NULL.
 * Every pointer may be device memory or page-locked mapped host memory (pom_host_alloc / pom_host_alloc_near): the
 * kernel reads and writes host memory directly.  Enqueues only: results are valid after pom_batch_sync(b). */
/* pom_batch_step and pom_batch_observe_planes in ONE call: at the end of the tick (after an auto-reset, so that the
 * planes show the state the next action applies to) every env's observation for the agents in agent_mask is written.
 * obs_dev, agent_mask, view and the layout are those of pom_batch_observe_planes.  Envs that are frozen (done / invalid,
 * no auto-reset) are observed as they are.  The call queues the step kernel and, behind it, the observation kernel, which
 * starts with the records the step wrote last.  With POM_OBS_FUSED=1 in the environment when the handle is made, the
 * step kernel writes the planes itself from the records it still holds in shared memory (no second read of the record
 * array, no second launch) - measured slower on a B200: the slice buffers are held twice as long (DESIGN section 8). */
int  pom_batch_step_observe(pom_batch* b, const uint8_t* moves_dev, uint32_t flags, uint8_t* obs_dev, uint32_t agent_mask, int view);
typedef struct pom_step_compact_io {
    const uint16_t* joint;
    uint32_t*       done_bits;
    uint32_t*       fin_env;
    uint8_t*        fin_status;
    uint32_t*       fin_count;
    uint32_t        fin_capacity;
    /* optional: observation planes written by the same call (see pom_batch_step_observe): DEVICE buffer, agents, window */
    uint8_t*        obs_dev;
    uint32_t        obs_agent_mask;
    int32_t         obs_view;
} pom_step_compact_io;
int  pom_batch_step_compact(pom_batch* b, const pom_step_compact_io* io, uint32_t flags);
/* pom_batch_step that also writes every env's per-agent REWARD of this tick, from inside the step kernel, for a learning
 * loop that keeps everything on the device (pom_batch_policy_moves -> pom_batch_step_rewards -> pom_batch_observe_planes).
 *   moves_dev  as for pom_batch_step
 *   rewards    n_envs x 4 int8 (4-byte aligned), required: byte a of env e at 4 e + a is the reward r[a] of agent a
 *   status     n_envs bytes or NULL: the end-of-tick status byte before any auto-reset, as pom_batch_step_host's status_host
 * Every env gets its four values, zeros included.  The reference has no reward; this is the project's definition, after the
 * reward function of the Pommerman Python environment.  With `stepped` = the env had neither DONE nor INVALID when the
 * tick started, `st` = its status byte as reported in `status`, and dead[a] = agent a's dead flag after the tick, the
 * first matching case decides:
 *     case                        free-for-all                      team game (POM_INIT_TEAMS)
 *     not stepped                 0 0 0 0                           0 0 0 0
 *     st & INVALID                0 0 0 0 (aborted, no outcome)     0 0 0 0
 *     DONE, not DRAW, winner w    +1 for agent w, -1 for the rest   +1 for both agents of team w, -1 for the other two
 *     DONE | DRAW                 -1 -1 -1 -1                       -1 -1 -1 -1
 *     TRUNCATED                   -1 -1 -1 -1                       -1 -1 -1 -1
 *     running                     -1 if dead[a], else 0             0 0 0 0
 * TRUNCATED is set only when DONE is not, so a win on the last allowed tick is a win.  In free-for-all a dead agent
 * collects -1 on every tick until its episode ends, the terminal tick included; a caller that wants a single -1 at death
 * takes the first one.  Frozen envs (done or invalid without POM_STEP_AUTORESET) get zeros.
 * Each pointer may be device memory or page-locked mapped host memory (pom_host_alloc).  Accepted flags: POM_STEP_AUTORESET,
 * POM_STEP_COUNT, POM_STEP_CONTINUE_UNDEFINED; states, counters, episode numbers and resets are those of pom_batch_step
 * with the same moves.  POM_E_ARG for any other flag (POM_STEP_RAW keeps no episode, so there is no outcome), a null
 * rewards, pageable buffers, or a handle made with POM_STEP_KERNEL=tile.  Enqueues only: results are valid after
 * pom_batch_sync(b). */
int  pom_batch_step_rewards(pom_batch* b, const uint8_t* moves_dev, uint32_t flags, int8_t* rewards, uint8_t* status);
/* The tick of pom_batch_step_rewards with the TEAM RADIO, on a handle made with POM_INIT_RADIO (POM_E_ARG otherwise).  The
 * reference has no radio; this is the project's definition, after Pommerman's team-radio environment (action space
 * Tuple(Discrete(6), Discrete(8), Discrete(8)): a move and two words).
 *   moves_dev  as for pom_batch_step
 *   msgs       n_envs x 4 bytes (4-byte aligned): byte a of env e at 4 e + a is agent a's message w0 | w1 << 3, two words
 *              w0, w1 of 0..7; bits 6..7 are ignored (as a joint action >= 1296 is taken modulo 6 per digit)
 *   rewards    n_envs x 4 int8 (4-byte aligned) or NULL, status  n_envs bytes or NULL: those of pom_batch_step_rewards
 * Each env keeps one LAST MESSAGE per agent (initially (0, 0)), in the record's padding bytes (pom_record.h), so the radio
 * moves no byte of state beyond the record.  Per env, together with its tick:
 *   not stepped (DONE or INVALID when the tick starts)   the messages stay as they are
 *   stepped      agent a's last message becomes msgs[4 e + a] & 63 if a was alive when the tick started, (0, 0) if it
 *                was dead (Pommerman's `not agent.is_alive` check before stepping): an agent that dies in this tick
 *                still gets its message through
 *   the env ended this tick and POM_STEP_AUTORESET re-initialised it: (0, 0) for everyone in the new episode
 * States, status bytes, counters and rewards are exactly those of pom_batch_step_rewards with the same moves: the radio
 * never changes the game.  Accepted flags: POM_STEP_AUTORESET, POM_STEP_COUNT, POM_STEP_CONTINUE_UNDEFINED.  POM_E_ARG for
 * any other flag, null moves or msgs, pageable buffers, misaligned msgs or rewards, or a handle made with
 * POM_STEP_KERNEL=tile.  Enqueues only: results are valid after pom_batch_sync(b).
 * Messages are env state, like the record.  Only this call, pom_batch_radio_upload and (re-)initialisation change them;
 * (re-)initialisation (auto-reset in any stepping path, pom_batch_reset, pom_batch_upload) sets (0, 0).  Every other call
 * - pom_batch_step[_host|_compact|_seq|_observe], pom_batch_rollout, pom_batch_policy_* - leaves the messages of running
 * envs as they were; pom_batch_clone copies them and pom_batch_expand_step children inherit their root's.  (Pommerman
 * sends (0, 0) for an action without words; here a step without messages keeps the last ones, which leaves every other
 * kernel as it is.)
 * The observation planes of a radio handle carry, for observer a, the last message of its teammate a ^ 2: byte 493 = w0
 * and byte 494 = w1 in the full layout, scalar bytes 9 and 10 in the cropped one (zero on every other handle); the radio
 * is not fogged.  This holds for pom_batch_observe_planes[_cropped], pom_batch_step_observe and pom_step_compact_io's
 * obs_dev; on a radio handle the last two always queue the observation kernel behind the step (POM_OBS_FUSED does not
 * apply).  pom_batch_observe (pom_state has no field for it) and the device SimpleAgent ignore the radio. */
int  pom_batch_step_radio(pom_batch* b, const uint8_t* moves_dev, const uint8_t* msgs, uint32_t flags, int8_t* rewards, uint8_t* status);
/* last messages of envs [first, first + count) of a radio handle (POM_E_ARG otherwise), count x 4 bytes of HOST memory in
 * the msgs encoding of pom_batch_step_radio; the upload ignores bits 6..7.  For fixtures, tree-search bookkeeping, tests. */
int  pom_batch_radio_download(pom_batch* b, uint64_t first, uint64_t count, uint8_t* msgs_host);
int  pom_batch_radio_upload(pom_batch* b, uint64_t first, uint64_t count, const uint8_t* msgs_host);
/* `ticks` fused ticks with the boards resident in shared memory; actions from pom_rng_moves(rng_seed,
 * global env index, tick0 + k); auto-reset unless POM_ROLL_NO_RESET.  Replaces the loop of
 * Environment::StartGame (environment.cpp:68-88) with RandomAgent/HarmlessAgent::act (bboard.hpp:517-533), or with
 * SimpleAgent::act for the agents named by POM_ROLL_SIMPLE(mask) (their draw: byte a of pom_rng_moves(.., 5)). */
int  pom_batch_rollout(pom_batch* b, uint32_t ticks, uint64_t rng_seed, uint32_t tick0, uint32_t flags);
/* the fused kernel with the CALLER's moves: `ticks` ticks in one launch, moves_dev = DEVICE pointer to ticks x n_envs x 4
 * bytes, tick-major (tick k, env e, agent a at ((k * n_envs) + e) * 4 + a).  The boards stay in shared memory for the
 * whole sequence, so the state crosses HBM once per launch instead of once per tick: the way to replay traces or to
 * evaluate fixed action plans in a search.  Same episode rule as the rollout: truncation at max_ticks, statistics,
 * auto-reset unless POM_ROLL_NO_RESET (the only flag accepted).  moves_dev may also point into page-locked mapped host
 * memory (pom_host_alloc): the kernel then fetches the moves over PCIe while it runs. */
int  pom_batch_step_seq(pom_batch* b, const uint8_t* moves_dev, uint32_t ticks, uint32_t flags);

/* ---- the reference's heuristic agent as a device-side action source (agents::SimpleAgent, simple_agent.cpp:12-141;
 *      bboard::strategy, strategy.cpp:37-338): the caller of the step path in Environment::Step
 *      (environment.cpp:137-146) and in the reference's benchmark.
 * For every running env and every agent a in agent_mask (bit a), byte a of moves_dev[env] <- SimpleAgent::act(state);
 * IDLE for a dead agent; bytes of agents outside the mask are kept, so a caller can mix its own moves with device
 * opponents.  The agent's one random draw per act is byte a of pom_rng_moves(seed, env_offset + env, tick, 5).
 * The agents' memories (pom_simple_agent, 8 bytes per agent) live on the device; they start zeroed and are zeroed
 * again when their env starts a new episode.  Follow with pom_batch_step(b, moves_dev, ...). */
int  pom_batch_policy_moves(pom_batch* b, uint8_t* moves_dev, uint64_t seed, uint32_t tick, uint32_t agent_mask);
/* same with HOST moves (n_envs x 4 bytes, read and written): upload, act, download, synchronise */
int  pom_batch_policy_moves_host(pom_batch* b, uint8_t* moves_host, uint64_t seed, uint32_t tick, uint32_t agent_mask);
/* SimpleAgent::act (simple_agent.cpp:128-141) for ONE agent of ONE env with the caller's own draw (0..4); the move
 * (0..5) goes to *move_out, the agent's memory on the device is updated.  For the bboard host mirror and tests. */
int  pom_batch_policy_act(pom_batch* b, uint64_t env, int agent, int draw, int* move_out);
int  pom_batch_policy_reset(pom_batch* b);                          /* all agents forget (new SimpleAgent objects) */
/* agent memories of envs [first, first+count) as count x 4 pom_simple_agent (HOST memory) */
int  pom_batch_policy_download(pom_batch* b, uint64_t first, uint64_t count, pom_simple_agent* out);
int  pom_batch_policy_upload(pom_batch* b, uint64_t first, uint64_t count, const pom_simple_agent* in);

/* Fog of war for the device SimpleAgent.  With a policy view v >= 0 every act of agent a is
 *     SimpleAgent::act( N_a( fog_state(state, a, v) ) )
 * where fog_state is the fogged State of pom_batch_observe (the unclamped square window [x - v, x + v] x [y - v, y + v]
 * around the agent's stored position: cells outside it become FOG, bombs outside it or off the board are dropped, other
 * agents outside it or dead are hidden with x = y = -1), and N_a makes every hidden agent absent: dead, at (0, 0) (as
 * SimpleActOnDevice does for the host agents of BatchEnvironment::SetViewRange).  The agent is otherwise the same one,
 * quirks included, team-aware on a team handle; its draw and its memory are those of the full-state agent.  It never reads
 * the flame queue.  So an enemy outside the window is not hunted or bombed and a bomb outside it does not make the agent
 * flee; with v = 0 the agent sees only its own cell.
 * The view is a property of the handle that may change between calls; it applies to every call made after it that runs
 * the device SimpleAgent: pom_batch_policy_moves[_host], pom_batch_rollout with POM_ROLL_SIMPLE (the fused and the
 * tick-by-tick path), pom_batch_policy_act.  A negative view (the default, -1) means the full state: the agent of the calls
 * above.  Any view >= 0 is accepted; from 15 on the window holds every position.  pom_batch_clone and
 * pom_batch_expand_step do not look at it.  The getter writes the view last set to *view_out. */
int  pom_batch_set_policy_view(pom_batch* b, int view);
int  pom_batch_get_policy_view(const pom_batch* b, int* view_out);

/* state copy for tree search (the reference copies the POD State by assignment, README.md:4):
 * dst env first_dst + i <- src env src_idx[i] (HOST array of n_dst indices).  dst may equal src.    */
int  pom_batch_clone(pom_batch* dst, uint64_t first_dst, const pom_batch* src, const uint32_t* src_idx, uint64_t n_dst);
/* tree-search expansion: child c = i * fanout + j of root src_idx[i] gets joint action j with
 * a_k = (j / 6^k) % 6 and is stepped once (clone + Step fused, one HBM write per child).
 * fanout <= 1296; dst needs n_roots * fanout envs; dst envs behind the last child are left untouched.
 * Enqueues on dst's stream (src_idx has been read when the call returns); work queued on src afterwards waits for it. */
int  pom_batch_expand_step(pom_batch* dst, const pom_batch* src, const uint32_t* src_idx, uint64_t n_roots, uint32_t fanout, uint32_t flags);

/* ---- State primitives on ONE env, executed by the device code of the step path (fixtures, the
 *      bboard::State host mirror).  a0..a2 depend on op:
 *      POM_OP_SPAWN_FLAME  x, y, strength   State::SpawnFlame     (bboard.cpp:198-263)
 *      POM_OP_EXPLODE_TOP  -                State::ExplodeTopBomb (bboard.cpp:191-196)
 *      POM_OP_EXPLODE_AT   index            State::ExplodeBombAt  (bboard.cpp:111-118)
 *      POM_OP_POP_FLAME    -                State::PopFlame       (bboard.cpp:148-180)          ---- */
enum { POM_OP_SPAWN_FLAME = 0, POM_OP_EXPLODE_TOP = 1, POM_OP_EXPLODE_AT = 2, POM_OP_POP_FLAME = 3 };
int  pom_batch_apply(pom_batch* b, uint64_t env, int op, int a0, int a1, int a2);
int  pom_batch_spawn_flame(pom_batch* b, uint64_t env, int x, int y, int strength);

/* InitBoardItems(state, seed) (bboard.cpp:346-382) for one seed, generated on `device`: fills board of a
 * zero-initialised State (agents are NOT placed).  *dirty = 1 when the seed hits the reference's
 * uninitialised read (the board is then whatever the draw sequence produced up to that point).          */
int  pom_make_board(int device, int32_t seed, pom_state* out, int* dirty);

/* ---- results ---- */
int  pom_batch_status(pom_batch* b, uint64_t first, uint64_t count, uint8_t* status_host);
int  pom_batch_stats(pom_batch* b, pom_stats* out);            /* synchronises */
int  pom_batch_clear_stats(pom_batch* b);

/* ---- action source shared by host and device ---- */
/* four moves packed little-endian, each mulhi16(x, n_actions), from splitmix64(seed, env, tick) */
uint32_t pom_rng_moves(uint64_t seed, uint64_t env, uint32_t tick, uint32_t n_actions);
/* fills a DEVICE buffer of n_envs x 4 bytes with pom_rng_moves(seed, env_offset + e, tick, n_actions) */
int  pom_batch_generate_moves(pom_batch* b, uint8_t* moves_dev, uint64_t seed, uint32_t tick, uint32_t n_actions);

/* ---- plumbing for callers that own CUDA objects (bench, NCCL reduce) ---- */
uint64_t pom_batch_size(const pom_batch* b);
int      pom_batch_device(const pom_batch* b);
void*    pom_batch_stream(const pom_batch* b);          /* cudaStream_t                           */
void*    pom_batch_stats_device_ptr(const pom_batch* b);/* POM_STATS_WORDS x uint64 on the device  */
void*    pom_batch_records_device_ptr(const pom_batch* b);
int      pom_device_alloc(int device, uint64_t bytes, void** out);
int      pom_device_free(int device, void* p);
/* either side may be host or device memory.  A plain synchronous cudaMemcpy on the default stream: it is NOT ordered
 * after work queued on a handle (handles use non-blocking streams) - call pom_batch_sync(b) first when the source is
 * being written by a queued call such as pom_batch_observe_planes. */
int      pom_device_copy(int device, void* dst, const void* src, uint64_t bytes);
int      pom_host_alloc(uint64_t bytes, void** out);    /* pinned host memory for pom_batch_step_host */
int      pom_host_free(void* p);
/* pinned host memory placed on the NUMA node of `device` (first touched by a thread bound to the CPUs that
 * /sys/bus/pci/devices/<gpu>/local_cpulist names), so that the kernel's zero-copy reads and writes do not cross the
 * inter-socket link; falls back to pom_host_alloc when the topology cannot be read.  Free with pom_host_free. */
int      pom_host_alloc_near(int device, uint64_t bytes, void** out);
/* binds the CALLING thread to the CPUs local to `device` (launch latency, polling of mapped buffers); returns POM_OK
 * also when the topology cannot be read (nothing is changed then) */
int      pom_bind_thread_near(int device);
/* timing helper: runs fn-less CUDA-event brackets on the handle's stream */
int      pom_batch_event_record(pom_batch* b, int which /* 0 = start, 1 = stop */);
int      pom_batch_event_elapsed_ms(pom_batch* b, float* ms);   /* synchronises on the stop event */
/* writes `bytes` of zeros to a scratch buffer larger than L2 (between timed iterations)          */
int      pom_batch_flush_l2(pom_batch* b);
/* number of kernels this library has launched on the handle (for bench.py's gpu_launches)        */
uint64_t pom_batch_launch_count(const pom_batch* b);

#ifdef __cplusplus
}
#endif
#endif /* POM_BATCH_H_ */
