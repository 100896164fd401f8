/*
 * pom_bboard.cpp — implementation of include/pom_bboard.hpp: the reference's bboard API surface on top
 * of the C ABI.  Field setters are host code (they are plain writes in the reference as well); everything
 * that advances the game goes to the GPU.  No CPU stepping path exists here.
 */
#include "pom_bboard.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <random>
#include <stdexcept>
#include <string>

namespace bboard
{

namespace
{

void check(int rc, const char* what)
{
    if(rc != POM_OK) throw std::runtime_error(std::string(what) + ": " + pom_last_error());
}

int default_device()
{
    const char* e = std::getenv("POM_DEVICE");
    return e ? std::atoi(e) : 0;
}

/* per-thread scratch batch used by the single-state and StepBatch calls; grows on demand */
struct Scratch
{
    pom_batch* h = nullptr;
    size_t cap = 0;
    ~Scratch() { if(h) pom_batch_destroy(h); }
    pom_batch* get(size_t n)
    {
        if(!h || cap < n)
        {
            if(h) pom_batch_destroy(h);
            h = nullptr;
            pom_init_desc d;
            std::memset(&d, 0, sizeof(d));
            d.n_templates = 1;
            d.first_seed = 0x1337;
            d.flags = POM_INIT_EMPTY;
            check(pom_batch_init(&h, default_device(), n, &d), "pom_batch_init");
            cap = n;
        }
        return h;
    }
};
thread_local Scratch scratch;

inline pom_state* raw(State* s) { return reinterpret_cast<pom_state*>(s); }

void apply(State* s, int op, int a0 = 0, int a1 = 0, int a2 = 0)
{
    pom_batch* h = scratch.get(1);
    check(pom_batch_upload(h, 0, 1, raw(s), nullptr), "pom_batch_upload");
    check(pom_batch_apply(h, 0, op, a0, a1, a2), "pom_batch_apply");
    check(pom_batch_download(h, 0, 1, raw(s), nullptr), "pom_batch_download");
}

}

/* SimpleAgent::act on the device for one host State: upload, act, fetch the move and the agent's memory */
int SimpleActOnDevice(const State* s, int id, pom_simple_agent* memory, int draw)
{
    pom_batch* h = scratch.get(1);
    /* A fogged State (BatchEnvironment::SetViewRange, pom_batch_observe) carries x = y = -1 for agents out of sight or
     * dead, which the packed record cannot hold.  Such an agent is not exposed to the observer (bboard.hpp:218-226), so
     * for the policy it is absent: marked dead at (0, 0), where nothing of the policy looks at it. */
    State seen = *s;
    for(int a = 0; a < AGENT_COUNT; a++)
    {
        AgentInfo& g = seen.agents[a];
        if(a != id && (g.x < 0 || g.y < 0 || g.x >= BOARD_SIZE || g.y >= BOARD_SIZE))
        {
            g.x = 0; g.y = 0; g.dead = true;
        }
    }
    /* likewise a visible flame cell whose flame started out of sight has lost its queue entry: for the policy it is just
     * a burning cell (the literal Item::FLAMES, which the record carries as an orphan flame) */
    for(int y = 0; y < BOARD_SIZE; y++)
    {
        for(int x = 0; x < BOARD_SIZE; x++)
        {
            const int v = seen.board[y][x];
            if(!IS_FLAME(v)) continue;
            const Position origin = { FLAME_ID(v) % BOARD_SIZE, FLAME_ID(v) / BOARD_SIZE };
            bool listed = false;
            for(int k = 0; k < seen.flames.count && !listed; k++) listed = seen.flames[k].position == origin;
            if(!listed) seen.board[y][x] = Item::FLAMES;
        }
    }
    check(pom_batch_upload(h, 0, 1, reinterpret_cast<const pom_state*>(&seen), nullptr), "pom_batch_upload");
    pom_simple_agent four[4];
    std::memset(four, 0, sizeof(four));
    four[id] = *memory;
    check(pom_batch_policy_upload(h, 0, 1, four), "pom_batch_policy_upload");
    int move = 0;
    check(pom_batch_policy_act(h, 0, id, draw, &move), "pom_batch_policy_act");
    check(pom_batch_policy_download(h, 0, 1, four), "pom_batch_policy_download");
    *memory = four[id];
    return move;
}

/* ---- State: field access (reference bboard.cpp:125-146, 265-333) ---- */
void State::PutAgent(int x, int y, int agentID)
{
    board[y][x] = Item::AGENT0 + agentID;
    agents[agentID].x = x;
    agents[agentID].y = y;
}

void State::PutAgentsInCorners(int a0, int a1, int a2, int a3)
{
    const int last = BOARD_SIZE - 1;
    board[0][0] = Item::AGENT0 + a0;
    board[0][last] = Item::AGENT0 + a1;
    board[last][last] = Item::AGENT0 + a2;
    board[last][0] = Item::AGENT0 + a3;
    /* like the reference, only the non-zero coordinates are written (a zeroed State is assumed) */
    agents[a1].x = agents[a2].x = last;
    agents[a2].y = agents[a3].y = last;
}

void State::PlantBomb(int x, int y, int id, bool setItem)
{
    PlantBombModifiedLife(x, y, id, BOMB_LIFETIME, setItem);
}

void State::PlantBombModifiedLife(int x, int y, int id, int lifeTime, bool setItem)
{
    AgentInfo& owner = agents[id];
    if(owner.bombCount >= owner.maxBombCount) return;
    Bomb& slot = bombs.NextPos();          /* direction / moved bits of the slot's previous tenant survive */
    SetBombID(slot, id);
    SetBombPosition(slot, x, y);
    SetBombStrength(slot, owner.bombStrength);
    SetBombTime(slot, lifeTime);
    if(setItem) board[y][x] = Item::BOMB;
    owner.bombCount++;
    bombs.count++;
}

int State::GetBombIndex(int x, int y)
{
    for(int i = 0; i < bombs.count; i++)
    {
        if(BMB_POS(bombs[i]) == x + (y << 4)) return i;
    }
    return -1;
}

bool State::HasBomb(int x, int y) { return GetBombIndex(x, y) >= 0; }

Bomb* State::GetBomb(int x, int y)
{
    const int i = GetBombIndex(x, y);
    return i < 0 ? nullptr : &bombs[i];
}

int State::GetAgent(int x, int y)
{
    for(int i = 0; i < AGENT_COUNT; i++)
    {
        if(!agents[i].dead && agents[i].x == x && agents[i].y == y) return i;
    }
    return -1;
}

Item State::FlagItem(int powFlag)
{
    switch(powFlag)
    {
        case 1: return Item::EXTRABOMB;
        case 2: return Item::INCRRANGE;
        case 3: return Item::KICK;
        default: return Item::PASSAGE;
    }
}

/* ---- State: game logic on the device ---- */
void State::SpawnFlame(int x, int y, int strength) { apply(this, POM_OP_SPAWN_FLAME, x, y, strength); }
void State::ExplodeTopBomb() { apply(this, POM_OP_EXPLODE_TOP); }
void State::ExplodeBombAt(int index) { apply(this, POM_OP_EXPLODE_AT, index); }
void State::PopFlame() { apply(this, POM_OP_POP_FLAME); }

void InitBoardItems(State& state, int seed)
{
    pom_state tmp;
    int dirty = 0;
    check(pom_make_board(default_device(), seed, &tmp, &dirty), "pom_make_board");
    if(dirty) throw std::runtime_error("InitBoardItems: this seed makes the reference read an uninitialised queue slot "
                                       "(bboard.cpp:351,367,372); choose another seed");
    std::memcpy(state.board, tmp.board, sizeof(state.board));
}

void InitState(State* state, int a0, int a1, int a2, int a3)
{
    InitBoardItems(*state);
    state->PutAgentsInCorners(a0, a1, a2, a3);
}

void StepBatch(State* states, const Move* moves, size_t n)
{
    if(n == 0) return;
    pom_batch* h = scratch.get(n);
    std::vector<uint8_t> mv(4 * n);
    for(size_t i = 0; i < 4 * n; i++) mv[i] = uint8_t(int(moves[i]));
    std::vector<uint8_t> zero(n, 0);
    check(pom_batch_upload(h, 0, n, raw(states), zero.data()), "pom_batch_upload");
    /* the scratch batch may be larger than n: the tail keeps whatever it held and its moves read as IDLE */
    std::vector<uint8_t> all(4 * pom_batch_size(h), 0);
    std::memcpy(all.data(), mv.data(), mv.size());
    check(pom_batch_step_host(h, all.data(), nullptr, POM_STEP_RAW), "pom_batch_step_host");
    std::vector<uint8_t> st(n);
    check(pom_batch_download(h, 0, n, raw(states), st.data()), "pom_batch_download");
    for(size_t i = 0; i < n; i++)
    {
        if(st[i] & POM_STATUS_INVALID)
            throw std::runtime_error("bboard::Step: the state left the reference's defined domain (the reference would crash or hang here)");
    }
}

void Step(State* state, Move* moves) { StepBatch(state, moves, 1); }

/* bboard.cpp:384-401 without the console output and the 80 ms sleep: every agent acts on the shared State (dead ones
 * too, as in the reference), then one Step; no early exit */
void StartGame(State* state, Agent* agents[AGENT_COUNT], int timeSteps)
{
    Move moves[AGENT_COUNT];
    for(int t = 0; t < timeSteps; t++)
    {
        for(int a = 0; a < AGENT_COUNT; a++) moves[a] = agents[a]->act(state);
        Step(state, moves);
    }
}

/* ---- Environment (reference environment.cpp:48-213) ---- */
Environment::Environment() : state(new State()), agents{{nullptr, nullptr, nullptr, nullptr}} {}
Environment::~Environment() {}

void Environment::MakeGame(std::array<Agent*, AGENT_COUNT> a, bool randomizePositions)
{
    InitBoardItems(*state);
    std::array<int, 4> order = {{0, 1, 2, 3}};
    if(randomizePositions)
    {
        std::random_device rd;
        std::mt19937 g(rd());
        std::shuffle(order.begin(), order.end(), g);
    }
    state->PutAgentsInCorners(order[0], order[1], order[2], order[3]);
    SetAgents(a);
    hasStarted = true;
}

void Environment::StartGame(int timeSteps, bool render, bool)
{
    state->timeStep = 0;
    while(!IsDone() && state->timeStep < timeSteps)
    {
        if(render && listener) listener(*this);
        Step(true);
    }
}

void Environment::Step(bool)
{
    if(!hasStarted || finished) return;
    Move m[AGENT_COUNT] = {Move::IDLE, Move::IDLE, Move::IDLE, Move::IDLE};
    for(int i = 0; i < AGENT_COUNT; i++)
    {
        if(!state->agents[i].dead)
        {
            m[i] = agents[i]->act(state.get());
            lastMoves[i] = m[i];
        }
    }
    bboard::Step(state.get(), m);
    state->timeStep++;
    if(state->aliveAgents == 1)
    {
        finished = true;
        for(int i = 0; i < AGENT_COUNT; i++) if(!state->agents[i].dead) agentWon = i;
    }
    if(state->aliveAgents == 0) { finished = true; isDraw = true; }
}

State& Environment::GetState() const { return *state; }
void Environment::SetAgents(std::array<Agent*, AGENT_COUNT> a)
{
    for(int i = 0; i < AGENT_COUNT; i++) a[size_t(i)]->id = i;
    agents = a;
}
Agent* Environment::GetAgent(unsigned agentID) const { return agents[agentID]; }
void Environment::SetStepListener(const std::function<void(const Environment&)>& f) { listener = f; }
bool Environment::IsDone() { return finished; }
bool Environment::IsDraw() { return isDraw; }
int Environment::GetWinner() { return agentWon; }
Move Environment::GetLastMove(int agentID) { return lastMoves[agentID]; }

/* ---- BatchEnvironment ---- */
BatchEnvironment::BatchEnvironment(size_t nGames, int device, uint64_t envOffset, uint32_t nTemplates, int firstSeed, uint32_t maxTicks,
                                   bool teams, bool radio)
    : n(nGames), teams(teams), radio(radio)
{
    pom_init_desc d;
    std::memset(&d, 0, sizeof(d));
    d.env_offset = envOffset;
    d.n_templates = nTemplates;
    d.first_seed = firstSeed;
    d.max_ticks = maxTicks;
    d.flags = (teams ? POM_INIT_TEAMS : 0) | (radio ? POM_INIT_RADIO : 0);
    check(pom_batch_init(&handle, device, n, &d), "pom_batch_init");
    movebuf.resize(4 * n);
}

BatchEnvironment::~BatchEnvironment() { if(handle) pom_batch_destroy(handle); }

void BatchEnvironment::MakeGames()
{
    check(pom_batch_reset(handle), "pom_batch_reset");
    check(pom_batch_sync(handle), "pom_batch_sync");
    fresh = false;
    tick = 0;
}

void BatchEnvironment::Refresh()
{
    if(fresh) return;
    host.resize(n);
    status.resize(n);
    check(pom_batch_download(handle, 0, n, reinterpret_cast<pom_state*>(host.data()), status.data()), "pom_batch_download");
    fresh = true;
}

size_t BatchEnvironment::Step(const Move* moves)
{
    for(size_t i = 0; i < 4 * n; i++) movebuf[i] = uint8_t(int(moves[i]));
    status.resize(n);
    check(pom_batch_step_host(handle, movebuf.data(), status.data(), 0), "pom_batch_step_host");
    fresh = false;
    tick++;
    size_t running = 0;
    for(size_t i = 0; i < n; i++) running += (status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID)) ? 0 : 1;
    return running;
}

std::vector<State> BatchEnvironment::Observe(int agentID, int view)
{
    std::vector<State> out(n);
    check(pom_batch_observe(handle, 0, n, agentID, view, reinterpret_cast<pom_state*>(out.data()), nullptr), "pom_batch_observe");
    return out;
}

size_t BatchEnvironment::Step(std::array<Agent*, AGENT_COUNT> agents)
{
    Refresh();
    std::vector<Move> mv(4 * n, Move::IDLE);
    for(int a = 0; a < AGENT_COUNT; a++)
    {
        std::vector<State> fogged;
        if(viewRange >= 0) fogged = Observe(a, viewRange);
        agents[size_t(a)]->id = a;
        for(size_t i = 0; i < n; i++)
        {
            if(status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID)) continue;
            if(!host[i].agents[a].dead) mv[4 * i + size_t(a)] = agents[size_t(a)]->act(viewRange >= 0 ? &fogged[i] : &host[i]);
        }
    }
    return Step(mv.data());
}

size_t BatchEnvironment::Step(const Move* moves, unsigned simpleMask, uint64_t seed)
{
    for(size_t i = 0; i < 4 * n; i++) movebuf[i] = uint8_t(int(moves[i]));
    if(simpleMask & 0xFu)
        check(pom_batch_policy_moves_host(handle, movebuf.data(), seed, tick, simpleMask & 0xFu), "pom_batch_policy_moves_host");
    status.resize(n);
    check(pom_batch_step_host(handle, movebuf.data(), status.data(), 0), "pom_batch_step_host");
    fresh = false;
    tick++;
    size_t running = 0;
    for(size_t i = 0; i < n; i++) running += (status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID)) ? 0 : 1;
    return running;
}

size_t BatchEnvironment::Step(const Move* moves, int8_t* rewards)
{
    /* one pinned buffer the kernel reads and writes directly: moves, rewards, status bytes */
    void* pinned = nullptr;
    check(pom_host_alloc(9 * n, &pinned), "pom_host_alloc");
    uint8_t* mv = static_cast<uint8_t*>(pinned);
    int8_t* rw = reinterpret_cast<int8_t*>(mv + 4 * n);
    uint8_t* st = mv + 8 * n;
    for(size_t i = 0; i < 4 * n; i++) mv[i] = uint8_t(int(moves[i]));
    int rc = pom_batch_step_rewards(handle, mv, 0, rw, st);
    if(rc == POM_OK) rc = pom_batch_sync(handle);
    if(rc == POM_OK)
    {
        std::memcpy(rewards, rw, 4 * n);
        status.assign(st, st + n);
    }
    pom_host_free(pinned);
    check(rc, "pom_batch_step_rewards");
    fresh = false;
    tick++;
    size_t running = 0;
    for(size_t i = 0; i < n; i++) running += (status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID)) ? 0 : 1;
    return running;
}

size_t BatchEnvironment::StepRadio(const Move* moves, const uint8_t* messages, int8_t* rewards)
{
    /* one pinned buffer the kernel reads and writes directly: moves, messages, rewards, status bytes */
    void* pinned = nullptr;
    check(pom_host_alloc(13 * n, &pinned), "pom_host_alloc");
    uint8_t* mv = static_cast<uint8_t*>(pinned);
    uint8_t* msg = mv + 4 * n;
    int8_t* rw = reinterpret_cast<int8_t*>(mv + 8 * n);
    uint8_t* st = mv + 12 * n;
    for(size_t i = 0; i < 4 * n; i++) mv[i] = uint8_t(int(moves[i]));
    std::memcpy(msg, messages, 4 * n);
    int rc = pom_batch_step_radio(handle, mv, msg, 0, rewards ? rw : nullptr, st);
    if(rc == POM_OK) rc = pom_batch_sync(handle);
    if(rc == POM_OK)
    {
        if(rewards) std::memcpy(rewards, rw, 4 * n);
        status.assign(st, st + n);
    }
    pom_host_free(pinned);
    check(rc, "pom_batch_step_radio");
    fresh = false;
    tick++;
    size_t running = 0;
    for(size_t i = 0; i < n; i++) running += (status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID)) ? 0 : 1;
    return running;
}

std::pair<int, int> BatchEnvironment::GetMessage(size_t i, int agent)
{
    uint8_t m[4];
    check(pom_batch_radio_download(handle, i, 1, m), "pom_batch_radio_download");
    const int v = m[agent & 3];
    return std::make_pair(v & 7, v >> 3);
}

size_t BatchEnvironment::StepSequence(const Move* moves, uint32_t ticks)
{
    const size_t bytes = size_t(ticks) * n * 4;
    void* pinned = nullptr;
    check(pom_host_alloc(bytes, &pinned), "pom_host_alloc");
    uint8_t* mv = static_cast<uint8_t*>(pinned);
    for(size_t i = 0; i < bytes; i++) mv[i] = uint8_t(int(moves[i]));
    int rc = pom_batch_step_seq(handle, mv, ticks, POM_ROLL_NO_RESET);     /* the kernel reads the pinned buffer directly */
    if(rc == POM_OK) rc = pom_batch_sync(handle);
    pom_host_free(pinned);
    check(rc, "pom_batch_step_seq");
    tick += ticks;
    fresh = false;
    Refresh();
    size_t running = 0;
    for(size_t i = 0; i < n; i++) running += (status[i] & (POM_STATUS_DONE | POM_STATUS_INVALID | POM_STATUS_TRUNCATED)) ? 0 : 1;
    return running;
}

void BatchEnvironment::SetSimpleViewRange(int view)
{
    check(pom_batch_set_policy_view(handle, view), "pom_batch_set_policy_view");
}

pom_stats BatchEnvironment::Rollout(uint32_t ticks, uint64_t seed, bool harmless, unsigned simpleMask)
{
    check(pom_batch_rollout(handle, ticks, seed, tick, (harmless ? POM_ROLL_HARMLESS : 0) | POM_ROLL_SIMPLE(simpleMask)), "pom_batch_rollout");
    tick += ticks;
    fresh = false;
    pom_stats s;
    check(pom_batch_stats(handle, &s), "pom_batch_stats");
    return s;
}

const std::vector<State>& BatchEnvironment::States() { Refresh(); return host; }
const std::vector<uint8_t>& BatchEnvironment::Status() { Refresh(); return status; }
bool BatchEnvironment::IsDone(size_t i) { Refresh(); return (status[i] & POM_STATUS_DONE) != 0; }
bool BatchEnvironment::IsDraw(size_t i) { Refresh(); return (status[i] & POM_STATUS_DRAW) != 0; }
int BatchEnvironment::GetWinner(size_t i)
{
    Refresh();
    if(teams || !(status[i] & POM_STATUS_DONE) || (status[i] & POM_STATUS_DRAW)) return -1;
    return (status[i] & POM_STATUS_WINNER_MASK) >> POM_STATUS_WINNER_SHIFT;
}
int BatchEnvironment::GetWinningTeam(size_t i)
{
    Refresh();
    if(!teams || !(status[i] & POM_STATUS_DONE) || (status[i] & POM_STATUS_DRAW)) return -1;
    return (status[i] & POM_STATUS_WINNER_MASK) >> POM_STATUS_WINNER_SHIFT;
}

}
