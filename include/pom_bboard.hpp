/*
 * pom_bboard.hpp — host-side C++ mirror of the reference's `bboard` step-path API on top of the
 * B200 batch engine (include/pom_batch.h).
 *
 * What it mirrors (reference dist1ll/pomcpp include/bboard.hpp): the constants (:15-27), Move/Direction
 * (:35-52), Item and its predicates (:54-109), FixedQueue (:115-188), Position (:192-196), AgentInfo
 * (:225-240), the Bomb word and its accessors (:261-335), Flame (:342-347), State with the methods the step
 * path and its tests use (:356-506), Agent (:517-533), Environment (:541-644), InitBoardItems / InitState /
 * Step (:651-668).  Names, argument meaning and the State layout (1004 bytes, same offsets) are the
 * reference's, so agent code written against it compiles unchanged and States can be exchanged with the
 * reference by plain copy.  Printing (PrintState/PrintItem, StartGame's console rendering) is out of scope
 * (SURVEY §2 rows 7, 14).  agents::SimpleAgent lives in pomcpp_b200/host/pom_agents.hpp; like Step it runs on the
 * device.
 *
 * What is different: nothing in here simulates on the CPU.  Field setters (PutItem, PutAgent, Kill,
 * PlantBomb, queue look-ups) are plain host writes/reads, exactly as in the reference; every function that
 * advances or explodes the game — Step, SpawnFlame, ExplodeTopBomb, ExplodeBombAt, PopFlame, InitBoardItems —
 * runs the CUDA device code of libpom_b200.so on the state (a one-env batch per host thread for the
 * single-state calls; use bboard::BatchEnvironment for throughput).  Without a GPU they throw
 * std::runtime_error("... no CPU fallback").
 *
 * Link with -lpom_b200 (pomcpp_b200/libpom_b200.so) and pomcpp_b200/host/libpom_host.a.
 */
#ifndef POM_BBOARD_HPP_
#define POM_BBOARD_HPP_

#include <array>
#include <cstdint>
#include <functional>
#include <iostream>
#include <memory>
#include <vector>

#include "pom_batch.h"
#include "pom_state.h"

namespace bboard
{

const int MOVE_COUNT = 4;
const int AGENT_COUNT = POM_AGENT_COUNT;
const int BOARD_SIZE = POM_BOARD_SIZE;
const int BOMB_LIFETIME = POM_BOMB_LIFETIME;
const int BOMB_DEFAULT_STRENGTH = POM_BOMB_DEFAULT_STRENGTH;
const int FLAME_LIFETIME = POM_FLAME_LIFETIME;
const int MAX_BOMBS_PER_AGENT = 5;
const int MAX_BOMBS = POM_MAX_BOMBS;

enum class Move { IDLE = 0, UP, DOWN, LEFT, RIGHT, BOMB };
enum class Direction { IDLE = 0, UP, DOWN, LEFT, RIGHT };

enum Item
{
    PASSAGE = POM_ITEM_PASSAGE, RIGID = POM_ITEM_RIGID, WOOD = POM_ITEM_WOOD, BOMB = POM_ITEM_BOMB,
    FLAMES = POM_ITEM_FLAMES, FOG = POM_ITEM_FOG, EXTRABOMB = POM_ITEM_EXTRABOMB,
    INCRRANGE = POM_ITEM_INCRRANGE, KICK = POM_ITEM_KICK, AGENTDUMMY = POM_ITEM_AGENTDUMMY,
    AGENT0 = POM_ITEM_AGENT0, AGENT1 = POM_ITEM_AGENT0 + 1, AGENT2 = POM_ITEM_AGENT0 + 2, AGENT3 = POM_ITEM_AGENT0 + 3
};

inline bool IS_WOOD(int x) { return (x >> 8) == 2; }
inline bool IS_POWERUP(int x) { return x > 5 && x < 9; }
inline bool IS_WALKABLE(int x) { return x == 0 || IS_POWERUP(x); }
inline bool IS_FLAME(int x) { return (x >> 16) == 4; }
inline bool IS_AGENT(int x) { return x >= (1 << 24); }
inline bool IS_STATIC_MOV_BLOCK(int x) { return x == 1 || IS_WOOD(x) || IS_POWERUP(x); }
inline int FLAME_ID(int x) { return (x & 0xFFFF) >> 3; }
inline int FLAME_POWFLAG(int x) { return x & 3; }
inline int WOOD_POWFLAG(int x) { return x & 3; }

template<typename T, int TSize>
struct FixedQueue
{
    T queue[TSize];
    int index = 0;
    int count = 0;

    int RemainingCapacity() { return TSize - count; }
    T& NextPos() { return queue[(index + count) % TSize]; }
    void AddElem(const T& e) { NextPos() = e; count++; }
    T& PopElem()
    {
        T& front = queue[index % TSize];
        index = (index + 1) % TSize;
        count--;
        return front;
    }
    void RemoveAt(int at)
    {
        for(int i = at + 1; i < count; i++)
        {
            const int from = (index + i) % TSize;
            queue[(from + TSize - 1) % TSize] = queue[from];
        }
        count--;
    }
    T& operator[](int offset) { return queue[(index + offset) % TSize]; }
    const T& operator[](int offset) const { return queue[(index + offset) % TSize]; }
};

struct Position { int x; int y; };
inline bool operator==(const Position& a, const Position& b) { return a.x == b.x && a.y == b.y; }
inline std::ostream& operator<<(std::ostream& out, const Position& p) { return out << '(' << p.x << ", " << p.y << ')'; }   /* bboard.hpp:203-207 */

struct AgentInfo
{
    int x;
    int y;
    int bombCount = 0;
    int maxBombCount = 1;
    int bombStrength = BOMB_DEFAULT_STRENGTH;
    bool canKick = false;
    bool dead = false;
    Position GetPos() { return {x, y}; }
};

typedef int Bomb;
inline int BMB_POS(Bomb b) { return b & 0xFF; }
inline int BMB_POS_X(Bomb b) { return b & 0xF; }
inline int BMB_POS_Y(Bomb b) { return (b >> 4) & 0xF; }
inline int BMB_ID(Bomb b) { return (b >> 8) & 0xF; }
inline int BMB_STRENGTH(Bomb b) { return (b >> 12) & 0xF; }
inline int BMB_TIME(Bomb b) { return (b >> 16) & 0xF; }
inline int BMB_DIR(Bomb b) { return (b >> 20) & 0xF; }
inline int BMB_MOVED(Bomb b) { return (b >> 24) & 0xF; }
/* the reference's setters are mask-and-ADD (a too-large value carries into the next field); kept */
inline void ReduceBombTimer(Bomb& b) { b = b - (1 << 16); }
inline void SetBombPosition(Bomb& b, int x, int y) { b = (b & ~0xFF) + x + (y << 4); }
inline void SetBombID(Bomb& b, int id) { b = (b & ~0xF00) + (id << 8); }
inline void SetBombStrength(Bomb& b, int s) { b = (b & ~0xF000) + (s << 12); }
inline void SetBombTime(Bomb& b, int t) { b = (b & ~0xF0000) + (t << 16); }
inline void SetBombDirection(Bomb& b, Direction d) { b = (b & ~0xF00000) + (int(d) << 20); }
inline void SetBombMovedFlag(Bomb& b, bool m) { b = (b & ~0xF000000) + (int(m) << 24); }

struct Flame
{
    Position position;
    int timeLeft = FLAME_LIFETIME;
    int strength;
};

struct State
{
    int board[BOARD_SIZE][BOARD_SIZE];
    int timeStep = 0;
    int aliveAgents = AGENT_COUNT;
    AgentInfo agents[AGENT_COUNT];
    FixedQueue<Bomb, MAX_BOMBS> bombs;
    FixedQueue<Flame, MAX_BOMBS> flames;

    int& operator[](const Position& p) { return board[p.y][p.x]; }

    /* plain field access, as in the reference */
    void PutItem(int x, int y, Item item) { board[y][x] = item; }
    void PutAgent(int x, int y, int agentID);
    void PutAgentsInCorners(int a0, int a1, int a2, int a3);
    void PlantBomb(int x, int y, int id, bool setItem = false);
    void PlantBombModifiedLife(int x, int y, int id, int lifeTime = BOMB_LIFETIME, bool setItem = false);
    bool HasBomb(int x, int y);
    Bomb* GetBomb(int x, int y);
    int GetAgent(int x, int y);
    int GetBombIndex(int x, int y);
    Item FlagItem(int powFlag);
    void Kill(int agentID)
    {
        if(!agents[agentID].dead) { agents[agentID].dead = true; aliveAgents--; }
    }
    template<typename... Args>
    void Kill(int agentID, Args... rest) { Kill(agentID); Kill(rest...); }

    /* game logic: executed by the device code (one-env batch of the calling thread) */
    void SpawnFlame(int x, int y, int strength);
    void ExplodeTopBomb();
    void ExplodeBombAt(int index);
    void PopFlame();
};
static_assert(sizeof(State) == sizeof(pom_state), "bboard::State must keep the reference layout");

struct Agent
{
    virtual ~Agent() {}
    int id = -1;
    virtual Move act(const State* state) = 0;
};

/* bboard.hpp:651-668 */
void InitBoardItems(State& state, int seed = 0x1337);
void InitState(State* state, int a0, int a1, int a2, int a3);
void Step(State* state, Move* moves);
/* bboard.hpp:677, bboard.cpp:384-401: `timeSteps` ticks of act() x 4 -> Step.  The reference also clears the console,
 * prints the board and sleeps 80 ms per tick; rendering is out of scope here, the game itself is identical. */
void StartGame(State* state, Agent* agents[AGENT_COUNT], int timeSteps);

/* agents::SimpleAgent::act for agent `id` on `state`, executed by the device policy code; `memory` is the agent's
 * persistent part, `draw` (0..4) its one random number.  Used by agents::SimpleAgent (pom_agents.hpp). */
int SimpleActOnDevice(const State* state, int id, pom_simple_agent* memory, int draw);

/* Many states at once: states[i] is advanced with moves[4*i .. 4*i+3]; one upload, one kernel, one download. */
void StepBatch(State* states, const Move* moves, size_t n);

/*
 * The reference's single-game Environment (bboard.hpp:541-644, environment.cpp:48-213) on top of the
 * batch engine.  Rendering and the 100 ms competitive collector thread are not mirrored: Step(true)
 * behaves like Step(false).
 */
class Environment
{
public:
    Environment();
    ~Environment();
    void MakeGame(std::array<Agent*, AGENT_COUNT> a, bool randomizePositions = false);
    void StartGame(int timeSteps, bool render = false, bool stepByStep = false);
    void Step(bool competitiveTimeLimit = false);
    State& GetState() const;
    void SetAgents(std::array<Agent*, AGENT_COUNT> agents);
    Agent* GetAgent(unsigned agentID) const;
    void SetStepListener(const std::function<void(const Environment&)>& f);
    bool IsDone();
    bool IsDraw();
    int GetWinner();
    Move GetLastMove(int agentID);

private:
    std::unique_ptr<State> state;
    std::array<Agent*, AGENT_COUNT> agents;
    std::function<void(const Environment&)> listener;
    bool finished = false, hasStarted = false, isDraw = false;
    int agentWon = -1;
    Move lastMoves[AGENT_COUNT];
};

/*
 * N independent games resident on one GPU: the batched counterpart of Environment, and the direct
 * caller of the hot path.  Actions come either from host Agent objects (act() is called on downloaded
 * States, as in Environment::Step) or from a caller-supplied move array; states stay on the device
 * between ticks.
 */
class BatchEnvironment
{
public:
    /* teams: the games are 2v2 team games (POM_INIT_TEAMS, include/pom_batch.h: agents 0 and 2 against 1 and 3) */
    BatchEnvironment(size_t nGames, int device = 0, uint64_t envOffset = 0, uint32_t nTemplates = 1024,
                     int firstSeed = 0x1337, uint32_t maxTicks = 0, bool teams = false);
    ~BatchEnvironment();
    BatchEnvironment(const BatchEnvironment&) = delete;
    BatchEnvironment& operator=(const BatchEnvironment&) = delete;

    size_t Size() const { return n; }
    /* all games back to their initial boards (InitState on clean seeds, agents 0..3 in the corners) */
    void MakeGames();
    /* one tick with the given moves (n x 4, host memory); returns the number of games still running */
    size_t Step(const Move* moves);
    /* one tick with actions from `agents` (shared by all games, called as agents[a]->act(&state_i) for every
     * live agent a of every running game i) */
    size_t Step(std::array<Agent*, AGENT_COUNT> agents);
    /* one tick in which the agents in simpleMask (bit a) are played by the device-side SimpleAgent
     * (simple_agent.cpp:12-141; their draws come from the shared counter RNG keyed by `seed`) and the others
     * take their move from `moves` (n x 4, host memory; entries of masked agents are ignored) */
    size_t Step(const Move* moves, unsigned simpleMask, uint64_t seed);
    /* Step(moves) that also fills rewards (n x 4, host memory) with every game's per-agent reward of this tick:
     * rewards[4 * i + a] for agent a of game i, as pom_batch_step_rewards defines it (include/pom_batch.h) */
    size_t Step(const Move* moves, int8_t* rewards);
    /* `ticks` ticks in ONE launch with the given moves (ticks x n x 4, tick-major, host memory); finished games freeze.
     * Returns the number of games still running.  For replaying traces and evaluating fixed action plans. */
    size_t StepSequence(const Move* moves, uint32_t ticks);
    /* `ticks` fused ticks on the device with auto-reset; agents in simpleMask play SimpleAgent, the others draw
     * uniformly (from {0..4} if harmless, else {0..5}); returns the counters */
    pom_stats Rollout(uint32_t ticks, uint64_t seed, bool harmless = false, unsigned simpleMask = 0);
    /* fog of war for the host agents of Step(agents): with view >= 0 every agent's act() receives the State as it sees it
     * through a square window of `view` cells (Pommerman: 4) — Item::FOG outside, agents / bombs / flames outside not
     * exposed (the "potentially fogged board state" of bboard.hpp:529, which the reference never implements);
     * view < 0 (default) = full observability, as in the reference */
    void SetViewRange(int view) { viewRange = view; }
    /* fog of war for the device SimpleAgent of Step(moves, simpleMask, seed) and Rollout(..., simpleMask): with view >= 0
     * it plays on what it sees through its window of `view` cells (pom_batch_set_policy_view); view < 0 (default) = the
     * full state.  Independent of SetViewRange, which applies to the host agents of Step(agents) only */
    void SetSimpleViewRange(int view);
    /* the State of every game as agent `agentID` observes it */
    std::vector<State> Observe(int agentID, int view);
    /* host copies */
    const std::vector<State>& States();
    const std::vector<uint8_t>& Status();          /* POM_STATUS_* per game */
    bool IsDone(size_t i);
    bool IsDraw(size_t i);
    int GetWinner(size_t i);                       /* the winning agent; -1 while running, on a draw and in a team game */
    bool IsTeamGame() const { return teams; }
    int GetWinningTeam(size_t i);                  /* team game: the winning team (0 or 1); -1 while running, on a draw */
    pom_batch* Handle() const { return handle; }

private:
    void Refresh();
    size_t n;
    pom_batch* handle = nullptr;
    std::vector<State> host;
    std::vector<uint8_t> status;
    std::vector<uint8_t> movebuf;
    bool fresh = false;
    uint32_t tick = 0;
    int viewRange = -1;
    bool teams = false;
};

}

namespace std
{
template<> struct hash<bboard::Position>                              /* bboard.hpp:694-703 */
{
    size_t operator()(const bboard::Position& p) const { return hash<int>()(p.x + p.y * bboard::BOARD_SIZE); }
};
}

#endif
