/*
 * pom_state.h — host-side array-of-structs view of ONE Pommerman env.
 *
 * This is the exchange format of the C ABI (pom_batch_upload / pom_batch_download)
 * and of the CPU oracle.  Its field order, sizes and offsets are those of the
 * reference's `bboard::State` (reference include/bboard.hpp:356-506, 1004 bytes:
 * board @0, timeStep @484, aliveAgents @488, agents @492, bombs @588, flames @676),
 * so a buffer of `pom_state` can be handed to code compiled against the reference
 * header (and the other way round) by plain copy.  Compare states FIELD-WISE:
 * `pom_agent` has two padding bytes (offsets 22-23) that carry no meaning.
 *
 * Plain C; no CUDA, no C++ types.
 */
#ifndef POM_STATE_H_
#define POM_STATE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* reference include/bboard.hpp:15-27 */
enum {
    POM_AGENT_COUNT     = 4,
    POM_BOARD_SIZE      = 11,
    POM_BOARD_CELLS     = 121,
    POM_BOMB_LIFETIME   = 10,
    POM_BOMB_DEFAULT_STRENGTH = 1,
    POM_FLAME_LIFETIME  = 4,
    POM_MAX_BOMBS       = 20
};

/* reference include/bboard.hpp:35-43 (Move) and :45-52 (Direction; first 5 identical) */
enum {
    POM_MOVE_IDLE = 0, POM_MOVE_UP = 1, POM_MOVE_DOWN = 2,
    POM_MOVE_LEFT = 3, POM_MOVE_RIGHT = 4, POM_MOVE_BOMB = 5
};

/* reference include/bboard.hpp:54-71 (Item): the 32-bit cell values of the AoS board */
enum {
    POM_ITEM_PASSAGE    = 0,
    POM_ITEM_RIGID      = 1,
    POM_ITEM_WOOD       = 2 << 8,     /* + powerup flag 0..4               */
    POM_ITEM_BOMB       = 3,
    POM_ITEM_FLAMES     = 4 << 16,    /* + ((x + 11*y) << 3) + powerup flag */
    POM_ITEM_FOG        = 5,
    POM_ITEM_EXTRABOMB  = 6,
    POM_ITEM_INCRRANGE  = 7,
    POM_ITEM_KICK       = 8,
    POM_ITEM_AGENTDUMMY = 9,
    POM_ITEM_AGENT0     = 1 << 24     /* + agent id 0..3 */
};

/* reference include/bboard.hpp:225-240 (AgentInfo), 24 bytes */
typedef struct pom_agent {
    int32_t x;
    int32_t y;
    int32_t bombCount;
    int32_t maxBombCount;
    int32_t bombStrength;
    uint8_t canKick;
    uint8_t dead;
    uint8_t _pad[2];
} pom_agent;

/* reference include/bboard.hpp:342-347 (Flame), 16 bytes */
typedef struct pom_flame {
    int32_t x;
    int32_t y;
    int32_t timeLeft;
    int32_t strength;
} pom_flame;

/* reference include/bboard.hpp:356-383 (State data members), 1004 bytes.
 * `bombs` holds the raw 32-bit bomb words (reference :261-335: bits 0-3 x, 4-7 y,
 * 8-11 owner, 12-15 strength, 16-19 time, 20-23 direction, 24-27 moved flag) in
 * PHYSICAL ring order; `*_index`/`*_count` are FixedQueue::index/count (:115-188). */
typedef struct pom_state {
    int32_t   board[POM_BOARD_SIZE][POM_BOARD_SIZE];   /* board[y][x] */
    int32_t   timeStep;
    int32_t   aliveAgents;
    pom_agent agents[POM_AGENT_COUNT];
    int32_t   bombs[POM_MAX_BOMBS];
    int32_t   bombs_index;
    int32_t   bombs_count;
    pom_flame flames[POM_MAX_BOMBS];
    int32_t   flames_index;
    int32_t   flames_count;
} pom_state;

/*
 * Persistent members of the reference's heuristic agent, agents::SimpleAgent (reference
 * include/agents.hpp:55-76), 8 bytes per agent, used by the device-side rollout policy
 * (include/pom_batch.h pom_batch_policy_moves / POM_ROLL_SIMPLE).  Everything else the agent holds
 * (`danger`, the reachability map `r`) is recomputed by every act(); its private mt19937_64 is replaced
 * by the shared counter RNG (one uniform{0..4} draw per agent and tick).
 *   recent[k]   recentPositions.queue[k] (PHYSICAL slot), x&15 | (y&15)<<4 with x,y in -1..11
 *               (a random move can point off the board, simple_agent.cpp:86,124-125); zero = (0,0), which
 *               is what a zero-initialised agent holds in its unwritten slots (read by _HasRPLoop, :24-35)
 *   rp_index    recentPositions.index   rp_count  recentPositions.count (0..4)
 *   move_queue  moveQueue.queue[4], 3 bits per slot; the slot beyond `count` is read when count == 1
 *               and the draw is odd (simple_agent.cpp:48,116), so stale contents are state
 */
typedef struct pom_simple_agent {
    uint8_t  recent[4];
    uint8_t  rp_index;
    uint8_t  rp_count;
    uint16_t move_queue;
} pom_simple_agent;

/* Per-env status byte kept next to the state by the batch engine.  The reference
 * keeps these in `Environment` (include/bboard.hpp:551-556, src/bboard/environment.cpp:150-168).
 * In the 2v2 team game (POM_INIT_TEAMS, pom_batch.h) a team is alive while one of its agents is not dead
 * (team 0 = agents 0 and 2, team 1 = agents 1 and 3): DONE when at most one team is alive, DRAW when none is,
 * and the winner field holds the winning TEAM index (0 or 1); with both teams alive the game goes on. */
enum {
    POM_STATUS_DONE        = 0x01,  /* Environment::finished                         */
    POM_STATUS_DRAW        = 0x02,  /* Environment::isDraw (aliveAgents == 0; team game: no team alive) */
    POM_STATUS_WINNER_MASK = 0x0C,  /* Environment::agentWon << 2 (valid if DONE&&!DRAW); team game: the team */
    POM_STATUS_WINNER_SHIFT = 2,
    POM_STATUS_INVALID     = 0x10,  /* env left the reference's defined domain (SURVEY §8c D3/D4,
                                       queue overflow, bad move byte): results undefined there too */
    POM_STATUS_TRUNCATED   = 0x20   /* rollout only: timeStep reached the tick limit  */
};

#ifdef __cplusplus
}
static_assert(sizeof(pom_state) == 1004, "pom_state must mirror bboard::State (1004 bytes)");
static_assert(sizeof(pom_agent) == 24, "pom_agent must mirror bboard::AgentInfo");
static_assert(sizeof(pom_simple_agent) == 8, "pom_simple_agent is 8 bytes");
#endif

#endif /* POM_STATE_H_ */
