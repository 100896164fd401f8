/*
 * pom_policy.cuh — the reference's heuristic agent as a device-side rollout policy.
 *
 * Re-states agents::SimpleAgent (reference src/agents/simple_agent.cpp:12-141) and the bboard::strategy helpers
 * it calls (src/bboard/strategy.cpp:37-338, include/strategy.hpp:134-168) on the packed record of pom_record.h:
 * one thread computes the move of one agent of its own env, reading the record in place.  It is the caller
 * of the step path in the reference's own benchmark (unit_test/bboard/performance_test.cpp:38,59-63).
 *
 * What is kept bit-exact: every decision of _Decide including the reference's quirks — the loop bounds of
 * MoveTowardsSafePlace (`y < radius`, strategy.cpp:130-132), SortDirections re-appending the element AFTER the
 * removed one (strategy.hpp:148-149), _HasRPLoop being vacuously true for fewer than two remembered positions
 * and reading an unwritten slot at two (simple_agent.cpp:24-35), moveQueue[1] being read when only one
 * direction is safe (:48,:125), paths ending at (but including) agent cells (strategy.cpp:44-52).
 *
 * What is restructured for the GPU:
 *   * the agent's persistent members are 8 bytes (pom_simple_agent, include/pom_state.h) instead of a 3 KB object;
 *     its private mt19937_64 is replaced by one caller-supplied draw in 0..4 per act (every path of _Decide
 *     consumes at most one intDist(rng));
 *   * FillRMap's queue BFS over a 121-int distance/predecessor map becomes 128-bit bitboard floods in registers
 *     (see "Bitboards" below): the map is only ever used for "is this cell reachable" and "what is the first move
 *     towards it", and both follow from flood fills; the tie-breaking of the FIFO queue is reproduced exactly;
 *   * the floods run lazily: only the two branches that read the map (danger > 0, enemy within 7) pay for them;
 *   * MoveTowardsSafePlace's double loop with an IsInDanger call per candidate becomes mask intersections and a
 *     find-first-set;
 *   * IsInDanger for the agent's cell and its four neighbours (the nine calls of _Decide + SafeDirections) is one
 *     pass over the bomb ring.
 *
 * Compiles as plain C++ too (POM_HD), so tests/hostsim can differential-test it on the CPU against the oracle.
 */
#ifndef POM_POLICY_CUH_
#define POM_POLICY_CUH_

#include "pom_core.cuh"

namespace pompolicy
{
using namespace pomcore;

/* persistent agent state, same bytes as pom_simple_agent: w0 = recent[4]; w1 = rp_index | rp_count<<8 | move_queue<<16 */
struct SimpleSt { uint32_t w0, w1; };

/* DesiredPosition on a nibble-packed position; x or y leaving the board wraps inside its own nibble (-1 -> 15, 11 stays 11) */
POM_HD uint32_t pos_step(uint32_t p, uint32_t m)
{
    const int d = move_delta(m);
    return (d & 15) ? ((p & 0xF0u) | (uint32_t(int(p) + d) & 15u)) : (uint32_t(int(p) + d) & 0xFFu);
}
POM_HD bool pos_oob(uint32_t p) { return (p & 15u) > 10u || (p >> 4) > 10u; }

/* IsInDanger (strategy.cpp:225-246) at (x, y), which may lie one cell off the board */
POM_HD uint32_t danger_at(const uint8_t* r, int x, int y)
{
    const int n = r[R_BCOUNT];
    uint32_t slot = r[R_BINDEX];
    uint32_t best = 16u;
    POM_LOOP
    for(int i = 0; i < n; i++)
    {
        const uint32_t b = reinterpret_cast<const uint32_t*>(r + R_BOMBS)[slot];
        slot = ring_next(slot);
        const int bx = int(b & 15u), by = int((b >> 4) & 15u), s = int((b >> 12) & 15u);
        const uint32_t t = (b >> 16) & 15u;
        const int dx = x - bx, dy = y - by;
        const bool hit = (dy == 0 && dx >= -s && dx <= s) || (dx == 0 && dy >= -s && dy <= s);   /* IsInBombRange, strategy.hpp:163-168 */
        if(hit && t < best) best = t;
    }
    return best == 16u ? 0u : best;
}

/* Fog of war for the policy (pom_batch_set_policy_view): the agent at (x, y) with view v >= 0 sees the square window
 * [x - v, x + v] x [y - v, y + v] of pomcore::fog_state / pom_oracle_fog.  A bomb is seen when its stored position lies
 * on the board and in the window (the fogged State drops the others). */
POM_HD bool in_view(int px, int py, int x, int y, int v)
{
    const int dx = px - x, dy = py - y;
    return dx >= -v && dx <= v && dy >= -v && dy <= v;
}
POM_HD bool bomb_in_view(uint32_t b, int x, int y, int v)
{
    const int bx = int(b & 15u), by = int((b >> 4) & 15u);
    return bx <= 10 && by <= 10 && in_view(bx, by, x, y, v);
}
/* The functions below take the view as a trailing argument pack `V... v`: one int in the FOG code, empty in the
 * full-state code, whose functions so keep the exact signatures (and the compiled code, register for register) they had
 * before fog existed.  view_of(v...) is the view, -1 without one. */
POM_HD int view_of() { return -1; }
POM_HD int view_of(int v) { return v; }
/* the same for a pack (x, y, v): the observer and its view */
POM_HD bool seen_by(int, int) { return true; }
POM_HD bool seen_by(int px, int py, int x, int y, int v) { return in_view(px, py, x, y, v); }

/* IsInDanger at DesiredPosition(x, y, m) for m = IDLE, UP, DOWN, LEFT, RIGHT: nibble m of the result.
 * FOG: only the bombs the agent at (x, y) sees with view `v` count */
template<bool FOG = false, class... V>
POM_HD uint32_t danger5(const uint8_t* r, int x, int y, V... v)
{
    const int n = r[R_BCOUNT];
    uint32_t slot = r[R_BINDEX];
    uint32_t b0 = 16u, b1 = 16u, b2 = 16u, b3 = 16u, b4 = 16u;
    POM_LOOP
    for(int i = 0; i < n; i++)
    {
        const uint32_t b = reinterpret_cast<const uint32_t*>(r + R_BOMBS)[slot];
        slot = ring_next(slot);
        if(FOG && !bomb_in_view(b, x, y, view_of(v...))) continue;
        const int s = int((b >> 12) & 15u);
        const uint32_t t = (b >> 16) & 15u;
        const int dx = x - int(b & 15u), dy = y - int((b >> 4) & 15u);
        const bool rowx = dx >= -s && dx <= s, coly = dy >= -s && dy <= s;
        if(((dy == 0 && rowx) || (dx == 0 && coly)) && t < b0) b0 = t;
        if(((dy == 1 && rowx) || (dx == 0 && dy - 1 >= -s && dy - 1 <= s)) && t < b1) b1 = t;       /* UP: y-1 */
        if(((dy == -1 && rowx) || (dx == 0 && dy + 1 >= -s && dy + 1 <= s)) && t < b2) b2 = t;      /* DOWN: y+1 */
        if(((dy == 0 && dx - 1 >= -s && dx - 1 <= s) || (dx == 1 && coly)) && t < b3) b3 = t;       /* LEFT: x-1 */
        if(((dy == 0 && dx + 1 >= -s && dx + 1 <= s) || (dx == -1 && coly)) && t < b4) b4 = t;      /* RIGHT: x+1 */
    }
    return (b0 & 15u) | ((b1 & 15u) << 4) | ((b2 & 15u) << 8) | ((b3 & 15u) << 12) | ((b4 & 15u) << 16);
}

POM_HD bool safe_condition(uint32_t danger, uint32_t min) { return danger == 0u || danger >= min; }   /* strategy.cpp:190-193 */

/* ---------------------------------------------------------------------------------------------
 * Bitboards: bit (x + 11*y) of a 128-bit word per cell.  FillRMap's queue BFS (strategy.cpp:58-95) visits
 * neighbours in the order down, up, right, left and is FIFO, so the path its predecessor chain encodes is the
 * lexicographically smallest (in that direction order) among the SHORTEST paths; MoveTowardsPosition
 * (strategy.cpp:101-124) only reports that path's first move.  Hence
 *     first move towards t  =  the first direction k in (down, up, right, left) whose neighbour s_k of the source
 *                              is nearest to t,
 * which a level-synchronous flood from t finds without storing distances or predecessors: grow the set from t
 * through walkable cells until it touches a neighbour of the source (stage B of simple_decide).  Every step of the flood is a handful of
 * 128-bit shifts and masks in registers, identical for all lanes of a warp, instead of a byte queue in local
 * memory with one divergent iteration per cell.
 * ------------------------------------------------------------------------------------------- */
typedef unsigned __int128 bb_t;

POM_HD bb_t bb_make(uint64_t hi, uint64_t lo) { return (bb_t(hi) << 64) | bb_t(lo); }
/* (a generic 128-bit shift by a variable amount is a dozen instructions and a branch; the two 64-bit halves are not) */
POM_HD bb_t bb_bit(int cell)
{
    const uint64_t one = 1ull << (cell & 63);
    return (cell & 64) ? bb_make(one, 0ull) : bb_make(0ull, one);
}
POM_HD int bb_lowest(bb_t b)           /* index of the lowest set bit, b != 0 */
{
    const uint64_t lo = uint64_t(b), hi = uint64_t(b >> 64);
#if defined(__CUDA_ARCH__)
    return lo ? __ffsll((long long)lo) - 1 : 63 + __ffsll((long long)hi);
#else
    return lo ? __builtin_ctzll(lo) : 64 + __builtin_ctzll(hi);
#endif
}

/* what the policy needs to know about the board, built once per env and tick for all four agents */
struct Boards {
    bb_t walk;      /* IS_WALKABLE: passage or powerup (bboard.hpp:87-90)        */
    bb_t agent;     /* item >= AGENT0: BFS paths may END here (strategy.cpp:44-52) */
};

POM_HD Boards make_boards(const uint8_t* r)
{
    Boards B;
    B.walk = 0; B.agent = 0;
    const uint32_t* w32 = reinterpret_cast<const uint32_t*>(r + R_BOARD);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int i = 0; i < 31; i++)
    {
        const uint32_t w = w32[i];
        /* per byte b < 0x80: MSB of (b + 0x80 - lo) is set iff b >= lo; flame bytes (MSB set) are masked out at the end */
        const uint32_t l = w & 0x7F7F7F7Fu, plain = ~w & 0x80808080u;
        const uint32_t ge1 = l + 0x7F7F7F7Fu, ge9 = l + 0x77777777u, ge12 = l + 0x74747474u, ge13 = l + 0x73737373u, ge17 = l + 0x6F6F6F6Fu;
        const uint32_t walk = (~ge1 | (ge9 & ~ge12)) & plain;       /* code 0 or 9..11 */
        const uint32_t agent = ge13 & ~ge17 & plain;                /* code 13..16     */
        /* the four byte flags -> one nibble (bit k = byte k) */
        const uint32_t wn = (((walk >> 7) * 0x01020408u) >> 24) & 15u;
        const uint32_t an = (((agent >> 7) * 0x01020408u) >> 24) & 15u;
        B.walk |= bb_t(wn) << (4 * i);
        B.agent |= bb_t(an) << (4 * i);
    }
    const bb_t full = bb_make(0x01FFFFFFFFFFFFFFull, 0xFFFFFFFFFFFFFFFFull);    /* word 30 also holds three non-board bytes */
    B.walk &= full;
    B.agent &= full;
    return B;
}

/* one flood step: everything in `pass` next to X joins X.  The column masks of the two horizontal shifts are folded
 * into pre-masked copies of `pass`, so a step is four 128-bit shifts, three ANDs and four ORs. */
struct Passable {
    bb_t any, from_left, from_right;   /* enterable at all / by a step to the right (not column 0) / to the left (not column 10) */
};
POM_HD Passable make_passable(bb_t pass)
{
    Passable P;
    P.any = pass;
    P.from_left = pass & bb_make(0x01FFBFF7FEFFDFFBull, 0xFF7FEFFDFFBFF7FEull);
    P.from_right = pass & bb_make(0x00FFDFFBFF7FEFFDull, 0xFFBFF7FEFFDFFBFFull);
    return P;
}
POM_HD bb_t flood_step(bb_t X, const Passable& P)
{
    return X | ((X << 1) & P.from_left) | ((X >> 1) & P.from_right) | (((X << 11) | (X >> 11)) & P.any);
}

/* cells in range of a bomb about to explode: IsInDanger(x, y) == 1, i.e. !_safe_condition(.., 2) (strategy.cpp:190-193,225-246).
 * FOG: only the bombs seen by the observer `obs` = (x, y, view) count */
template<bool FOG = false, class... V>
POM_HD bb_t unsafe_cells(const uint8_t* r, V... obs)
{
    const int n = r[R_BCOUNT];
    uint32_t slot = r[R_BINDEX];
    bb_t t1 = 0, t0 = 0;
    const bb_t col0 = bb_make(0x0000400801002004ull, 0x0080100200400801ull);
    POM_LOOP
    for(int i = 0; i < n; i++)
    {
        const uint32_t b = reinterpret_cast<const uint32_t*>(r + R_BOMBS)[slot];
        slot = ring_next(slot);
        const uint32_t t = (b >> 16) & 15u;
        if(t > 1u) continue;
        const int bx = int(b & 15u), by = int((b >> 4) & 15u), s = int((b >> 12) & 15u);
        if(bx > 10 || by > 10) continue;                          /* cannot cover a board cell's row AND column test */
        if(FOG && !seen_by(bx, by, obs...)) continue;
        const int x0 = bx - s < 0 ? 0 : bx - s, x1 = bx + s > 10 ? 10 : bx + s;
        const int y0 = by - s < 0 ? 0 : by - s, y1 = by + s > 10 ? 10 : by + s;
        const bb_t row = bb_t((2u << x1) - (1u << x0)) << (11 * by);
        const bb_t rows = (bb_bit(11 * (y1 + 1)) - 1) ^ (bb_bit(11 * y0) - 1);
        const bb_t cross = row | ((col0 << bx) & rows);
        if(t == 1u) t1 |= cross; else t0 |= cross;
    }
    return t1 & ~t0;                                              /* a covering bomb with time 0 makes the minimum 0 = "no danger" */
}

/* the board cells of the window of the agent at (x, y) with view v >= 0: a row band times a column band (the FOG
 * policy's view of the board, pomcore::fog_state: every cell outside it is FOG, neither walkable nor an agent cell) */
POM_HD bb_t view_cells(int x, int y, int v)
{
    const int x0 = x - v < 0 ? 0 : x - v, x1 = x + v > 10 ? 10 : x + v;
    const int y0 = y - v < 0 ? 0 : y - v, y1 = y + v > 10 ? 10 : y + v;
    const bb_t col0 = bb_make(0x0000400801002004ull, 0x0080100200400801ull);
    const bb_t cols = (col0 << (x1 + 1)) - (col0 << x0);         /* columns x0..x1 of every row: no borrow crosses a row */
    const bb_t rows = (bb_bit(11 * (y1 + 1)) - 1) ^ (bb_bit(11 * y0) - 1);
    return cols & rows;
}

/* the cells MoveTowardsSafePlace's double loop looks at (strategy.cpp:130-135): Manhattan distance <= radius and,
 * because the loops stop at `radius` instead of origin + radius (sic), x < radius and y < radius */
POM_HD bb_t safe_place_region(int ox, int oy, int radius)
{
    bb_t region = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int y = 0; y < 11; y++)
    {
        const int dy = y < oy ? oy - y : y - oy, h = radius - dy;
        int x0 = ox - h, x1 = ox + h;
        if(x0 < 0) x0 = 0;
        if(x1 > 10) x1 = 10;
        if(x1 > radius - 1) x1 = radius - 1;
        if(h >= 0 && y < radius && x0 <= x1) region |= bb_t((2u << x1) - (1u << x0)) << (11 * y);
    }
    return region;
}

/* the 3-bit slots of moveQueue.queue */
POM_HD uint32_t mq_get(uint32_t mq, int i) { return (mq >> (3 * (i & 3))) & 7u; }
POM_HD uint32_t mq_set(uint32_t mq, int i, uint32_t v) { const int s = 3 * (i & 3); return (mq & ~(7u << s)) | (v << s); }

/* _MoveSafeOneSpace / the tail of _Decide (simple_agent.cpp:37-49,113-126): SafeDirections (strategy.cpp:194-219)
 * + SortDirections (strategy.hpp:134-158) + the random pick among the first two.
 * blind: the neighbours are out of sight (FOG, view 0): FOG cells, none of them walkable */
template<bool FOG = false, class... V>
POM_HD uint32_t pick_safe_direction(const uint8_t* r, uint32_t pos, uint32_t dg, SimpleSt& st, uint32_t draw, V... blind)
{
    uint32_t mq = st.w1 >> 16;
    int count = 0;
    /* live slots of recentPositions: `count` physical slots starting at `index` (a byte mask, rotated into place) */
    const uint32_t rp_index = st.w1 & 3u, rp_count = (st.w1 >> 8) & 0xFFu;
    const uint32_t first = rp_count >= 4u ? 0x80808080u : (0x80808080u & ((1u << (8u * rp_count)) - 1u));
    const uint32_t live = (first << (8u * rp_index)) | (rp_index ? first >> (32u - 8u * rp_index) : 0u);
    uint32_t seen = 0;                                         /* bit mv: DesiredPosition(mv) was visited recently */
    POM_LOOP
    for(int k = 0; k < 4; k++)
    {
        const uint32_t mv = 4u - uint32_t(k);                  /* RIGHT, LEFT, DOWN, UP */
        const uint32_t p = pos_step(pos, mv);
        if(pos_oob(p) || (FOG && (blind || ...))) continue;
        if(!c_is_walkable(r[R_BOARD + cell_of(p)])) continue;
        if(!safe_condition((dg >> (4u * mv)) & 15u, 2u)) continue;
        mq = mq_set(mq, count, mv);
        count++;
        if(bytes_equal(st.w0, p) & live) seen |= 1u << mv;
    }
    const int moves = count;
    int removes = 0;
    POM_LOOP
    for(int i = 0; i < moves && removes < 4; i++)
    {
        if((seen >> mq_get(mq, i)) & 1u)
        {
            for(int k = i + 1; k < count; k++) mq = mq_set(mq, k - 1, mq_get(mq, k));   /* RemoveAt(i) */
            count--;
            mq = mq_set(mq, count, mq_get(mq, i));                                      /* AddElem(q[i]): the element AFTER it (sic) */
            count++;
            i--;
            removes++;
        }
    }
    st.w1 = (st.w1 & 0xFFFFu) | (mq << 16);
    if(count == 0) return POM_MOVE_IDLE;
    return mq_get(mq, int(draw & 1u));
}

/*
 * _Decide (simple_agent.cpp:52-127) for the four agents of an env, laid out so that the lanes of a warp stay
 * together where it is expensive.  The flood loops dominate the cost and only some agents need one (FLEE: danger > 0,
 * MoveTowardsSafePlace; HUNT: an enemy within 7 cells, MoveTowardsEnemy), with very different lengths.  So:
 *   phase 1  per agent: classify (plan_agent) — cheap, no floods;
 *   phase 2  ONE loop runs all flood jobs of the env back to back: a lane whose agent 0 needs no flood is already
 *            working on agent 2's while its neighbour still floods for agent 0.  The sum of an env's jobs varies far
 *            less between lanes than any single job, and there is exactly one copy of the flood step in the code;
 *   phase 3  per agent: finish the decision (finish_agent) and update the agent's memory (SimpleAgent::act).
 * The agents only read the state, so the order in which their decisions are evaluated does not matter.
 */
enum { K_NONE = 0, K_FLEE = 1, K_HUNT = 2 };

struct Plan {
    uint32_t dg;            /* IsInDanger at the agent's cell and its four neighbours, nibble per Move (danger5) */
    uint8_t  kind;          /* K_*                                                                              */
    uint8_t  target;        /* HUNT: cell of the enemy to walk towards, FLEE: filled by phase 2; 0xFF = none    */
    uint8_t  result;        /* move decided in phase 1, 0xFF = not yet                                          */
    uint8_t  wood_next;     /* "bomb the wood next to me" is still to be tried (:107-110)                        */
    uint8_t  move;          /* phase 2: first move towards the target (IDLE if there is none)                   */
    bb_t     region;        /* FLEE: the cells MoveTowardsSafePlace scans                                        */
};

/* phase 1: which branch of _Decide is agent `id` in.
 * TEAMS: the team game (env_post): the teammate id ^ 2 is no enemy - neither for IsAdjacentEnemy nor as the target of
 * MoveTowardsEnemy; everything else is the same agent.
 * FOG: the agent sees through the window of view v (in_view): bombs outside it do not count, and an enemy outside it
 * (Chebyshev distance > v) is absent, as a hidden agent of the fogged State is for SimpleActOnDevice */
template<bool TEAMS = false, bool FOG = false, class... V>
POM_HD Plan plan_agent(const uint8_t* r, int id, const SimpleSt& st, uint32_t draw, V... v)
{
    Plan pl;
    const uint32_t pos = r[R_APOS + id];
    const int x = int(pos & 15u), y = int(pos >> 4);
    pl.dg = danger5<FOG>(r, x, y, v...);
    pl.kind = K_NONE; pl.target = 0xFFu; pl.result = 0xFFu; pl.wood_next = 0; pl.move = POM_MOVE_IDLE;
    if((pl.dg & 15u) > 0u)
    {
        pl.kind = K_FLEE;
        pl.region = safe_place_region(x, y, int(pl.dg & 15u));
    }
    else if(int(int8_t(r[R_ABCNT + id])) < int(r[R_AMAX + id]))
    {
        /* IsAdjacentEnemy (strategy.cpp:296-312): nearest live enemy, Manhattan */
        int dmin = 99, target = -1;
        for(int i = 0; i < 4; i++)
        {
            if(i == id || (TEAMS && i == (id ^ 2)) || (r[R_AFLAGS + i] & AF_DEAD)) continue;
            if(FOG && !in_view(int(r[R_APOS + i] & 15u), int(r[R_APOS + i] >> 4), x, y, view_of(v...))) continue;
            const int dx = int(r[R_APOS + i] & 15u) - x, dy = int(r[R_APOS + i] >> 4) - y;
            const int d = (dx < 0 ? -dx : dx) + (dy < 0 ? -dy : dy);
            if(d < dmin) dmin = d;
            /* MoveTowardsEnemy (strategy.cpp:165-183) takes the FIRST agent within the radius that does not share
             * the source's cell */
            if(target < 0 && d <= 7 && d != 0) target = i;
        }
        if(dmin <= 1) pl.result = POM_MOVE_BOMB;
        else
        {
            pl.wood_next = 1;
            if(dmin <= 7)
            {
                /* _HasRPLoop, simple_agent.cpp:24-35 */
                const uint32_t rp_index = st.w1 & 0xFFu, rp_count = (st.w1 >> 8) & 0xFFu;
                bool loop = true;
                for(uint32_t i = 0; i < rp_count / 2u; i++)
                    loop = loop && byte_of(st.w0, int((rp_index + i) & 3u)) == byte_of(st.w0, int((rp_index + i + 2u) & 3u));
                if(loop) pl.result = uint8_t(draw & 3u);        /* Move(intDist(rng) % 4) */
                else
                {
                    pl.kind = K_HUNT;
                    if(target >= 0) pl.target = uint8_t(int(r[R_APOS + target] & 15u) + 11 * int(r[R_APOS + target] >> 4));
                }
            }
        }
    }
    return pl;
}

/* phase 2: the flood jobs of one env.
 *   job A (FLEE)  FillRMap's reachable set = flood from the source to a fixpoint (the BFS never re-enters its source,
 *                 and neither does the flood: the source is in the set from the start); then the first cell of
 *                 MoveTowardsSafePlace's scan (strategy.cpp:126-144) that is reachable and not about to blow up
 *                 becomes the target of a job B;
 *   job B         MoveTowardsPosition (strategy.cpp:101-124): grow a set from the target through walkable cells
 *                 until it touches a neighbour of the source; the neighbours touched first are the nearest to the
 *                 target, and the first of them in the order down, up, right, left is where FillRMap's path starts. */
POM_HD bool bb_test(bb_t b, int cell)
{
    const uint64_t half = (cell & 64) ? uint64_t(b >> 64) : uint64_t(b);
    return ((half >> (cell & 63)) & 1ull) != 0ull;
}

/* FOG: every job sees the board through its agent's window (view v): walkable and agent cells outside it are FOG, and
 * the unsafe cells come from the bombs that agent sees, so they are found per job instead of once per env */
template<bool FOG = false, class... V>
POM_HD void run_floods(const uint8_t* r, const Boards& B, Plan* pl, uint32_t jobs, V... v)
{
    /* jobs: bit a = agent a has a flood to run (FLEE, or HUNT with an enemy to walk to) */
    bb_t unsafe = 0;
    bool have_unsafe = false;
    int a = -1;
    bool mode_b = false;
    bb_t X = 0, src = 0;
    Passable P = make_passable(0);
    for(;;)
    {
        if(a >= 0)
        {
            /* the hot part: one flood step of the current job.  The source cell itself counts as passable: in job A
             * it is where the flood starts, in job B the flood reaching it is the stop condition. */
            const bb_t n = flood_step(X, P);
            const bool hit = mode_b && (n & src) != 0;
            if(!hit && n != X) { X = n; continue; }
            /* the job is over, or turns from A into B */
            const uint32_t pos = r[R_APOS + a];
            const int x = int(pos & 15u), y = int(pos >> 4), s = x + 11 * y;
            if(hit)
            {
                pl[a].move = uint8_t((y < 10 && bb_test(X, s + 11)) ? POM_MOVE_DOWN : (y > 0 && bb_test(X, s - 11)) ? POM_MOVE_UP :
                                     (x < 10 && bb_test(X, s + 1)) ? POM_MOVE_RIGHT : POM_MOVE_LEFT);
            }
            else if(mode_b)
            {
                /* unreachable target (HUNT only): its predecessor field is 0 = cell (0,0); a source standing ON (0,0)
                 * takes the "predecessor is the source" branch and walks towards the target's side, everybody else idles */
                pl[a].move = uint8_t(pos != 0u ? POM_MOVE_IDLE : (pl[a].target % 11u > 0u ? POM_MOVE_RIGHT : POM_MOVE_DOWN));
            }
            else
            {
                /* agent cells next to the flooded area are reached but not left (strategy.cpp:44-52) */
                const bb_t edge = ((X << 1) & bb_make(0x01FFBFF7FEFFDFFBull, 0xFF7FEFFDFFBFF7FEull)) |
                                  ((X >> 1) & bb_make(0x00FFDFFBFF7FEFFDull, 0xFFBFF7FEFFDFFBFFull)) | (X << 11) | (X >> 11);
                bb_t cand = (X | (edge & (FOG ? B.agent & view_cells(x, y, view_of(v...)) : B.agent))) & ~src & pl[a].region;
                if(cand != 0)
                {
                    if(!have_unsafe)
                    {
                        if constexpr(FOG) unsafe = unsafe_cells<FOG>(r, x, y, v...);
                        else unsafe = unsafe_cells(r);
                        have_unsafe = true;
                    }
                    cand &= ~unsafe;
                }
                if(cand != 0)
                {
                    const int t = bb_lowest(cand);               /* scan order of the reference: y outer, x inner */
                    pl[a].target = uint8_t(t);
                    X = bb_bit(t);
                    mode_b = true;
                    continue;
                }
            }
        }
        /* next job */
        if(jobs == 0u) break;
        a = (jobs & 1u) ? 0 : (jobs & 2u) ? 1 : (jobs & 4u) ? 2 : 3;
        jobs &= jobs - 1u;
        {
            const uint32_t pos = r[R_APOS + a];
            src = bb_bit(int(pos & 15u) + 11 * int(pos >> 4));
            if(FOG) have_unsafe = false;
            P = make_passable((FOG ? B.walk & view_cells(int(pos & 15u), int(pos >> 4), view_of(v...)) : B.walk) | src);
            mode_b = pl[a].kind == K_HUNT;
            /* FillRMap only ever enters walkable cells and agent cells (strategy.cpp:44-46): a target on anything else
             * (possible for an enemy only in hand-made states whose board and agent list disagree) is unreachable,
             * which an empty start set reports right away */
            const bb_t ends = FOG ? (B.walk | B.agent) & view_cells(int(pos & 15u), int(pos >> 4), view_of(v...)) : B.walk | B.agent;
            X = !mode_b ? src : (bb_test(ends, pl[a].target) ? bb_bit(pl[a].target) : bb_t(0));
        }
    }
}

/* phase 3: the rest of _Decide for agent `id`.  FOG: with view 0 the four neighbours are FOG (neither walkable nor wood);
 * with view >= 1 they are in sight, and the destination of a planned move is a neighbour or the agent's own cell */
template<bool FOG = false, class... V>
POM_HD uint32_t finish_agent(const uint8_t* r, int id, const Plan& pl, SimpleSt& st, uint32_t draw, V... v)
{
    const bool blind = FOG && view_of(v...) < 1;
    const uint32_t pos = r[R_APOS + id];
    uint32_t result = pl.result;
    /* take the move if its destination is walkable and safe enough (:62-66, :93-98) */
    if(pl.kind != K_NONE)
    {
        const uint32_t m = pl.move, p = pos_step(pos, m);
        if(!pos_oob(p) && (!blind || m == POM_MOVE_IDLE) && c_is_walkable(r[R_BOARD + cell_of(p)]) && safe_condition((pl.dg >> (4u * m)) & 15u, pl.kind == K_FLEE ? 2u : 5u)) result = m;
    }
    if(result == 0xFFu && pl.wood_next)
    {
        /* IsAdjacentItem(state, id, 1, WOOD), strategy.cpp:314-338: own cell and the four neighbours */
        bool wood = c_is_wood(r[R_BOARD + cell_of(pos)]);
        for(uint32_t mv = 1; mv <= 4u; mv++)
        {
            const uint32_t p = pos_step(pos, mv);
            if(!pos_oob(p) && !blind) wood = wood || c_is_wood(r[R_BOARD + cell_of(p)]);
        }
        if(wood) result = POM_MOVE_BOMB;
    }
    /* everybody who is still undecided moves one safe step (:68, :113-126) */
    if(result == 0xFFu) result = FOG ? pick_safe_direction<FOG>(r, pos, pl.dg, st, draw, blind) : pick_safe_direction(r, pos, pl.dg, st, draw);
    return result;
}

/* SimpleAgent::act's bookkeeping (simple_agent.cpp:128-141): remember where move m leads */
POM_HD void remember_position(const uint8_t* r, int id, SimpleSt& st, uint32_t m)
{
    const uint32_t p = pos_step(r[R_APOS + id], m);            /* BOMB and IDLE remember the agent's own cell */
    uint32_t idx = st.w1 & 0xFFu, cnt = (st.w1 >> 8) & 0xFFu;
    if(cnt == 4u) { idx = (idx + 1u) & 3u; cnt = 3u; }          /* PopElem when full */
    st.w0 = with_byte(st.w0, int((idx + cnt) & 3u), p);
    cnt++;
    st.w1 = (st.w1 & 0xFFFF0000u) | idx | (cnt << 8);
}

/* SimpleAgent::act for ONE agent.  FOG: the agent plays on what it sees through its window of view v >= 0 (in_view) */
template<bool TEAMS = false, bool FOG = false, class... V>
POM_HD uint32_t simple_act(const uint8_t* r, const Boards& B, int id, SimpleSt& st, uint32_t draw, V... v)
{
    Plan pl[4];
    for(int a = 0; a < 4; a++) pl[a].kind = K_NONE;
    pl[id] = plan_agent<TEAMS, FOG>(r, id, st, draw, v...);
    run_floods<FOG>(r, B, pl, (pl[id].kind == K_FLEE || pl[id].target != 0xFFu) ? 1u << id : 0u, v...);
    const uint32_t m = finish_agent<FOG>(r, id, pl[id], st, draw, v...);
    remember_position(r, id, st, m);
    return m;
}

/* Environment::Step's collection loop (environment.cpp:137-146) for the agents in `mask`: returns `moves` with the
 * bytes of the masked agents replaced (IDLE for a dead agent, whose slot the reference leaves unwritten).
 * `draws` = pom_rng_moves(seed, env, tick, 5): byte a is agent a's uniform{0..4} draw.  `S` gives access to the
 * four agent states: S.load(a) / S.store(a, st) (an array on the host, shared or global memory in the kernels).
 * FOG: every agent plays on what it sees through its own window of view v >= 0 (simple_act); the boards are built once
 * per env all the same and each agent's window is applied where it reads them. */
template<bool TEAMS = false, bool FOG = false, class Store, class... V>
POM_HD uint32_t simple_moves(const uint8_t* r, uint32_t mask, uint32_t moves, uint32_t draws, Store& S, V... v)
{
    const Boards B = make_boards(r);
    Plan pl[4];
    uint32_t jobs = 0;
    POM_LOOP
    for(int a = 0; a < 4; a++)
    {
        pl[a].kind = K_NONE;
        if(((mask >> a) & 1u) && !(r[R_AFLAGS + a] & AF_DEAD))
        {
            pl[a] = plan_agent<TEAMS, FOG>(r, a, S.load(a), byte_of(draws, a), v...);
            if(pl[a].kind == K_FLEE || pl[a].target != 0xFFu) jobs |= 1u << a;
        }
    }
    run_floods<FOG>(r, B, pl, jobs, v...);
    POM_LOOP
    for(int a = 0; a < 4; a++)
    {
        if(!((mask >> a) & 1u)) continue;
        uint32_t m = POM_MOVE_IDLE;
        if(!(r[R_AFLAGS + a] & AF_DEAD))
        {
            SimpleSt st = S.load(a);
            m = finish_agent<FOG>(r, a, pl[a], st, byte_of(draws, a), v...);
            remember_position(r, a, st, m);
            S.store(a, st);
        }
        moves = with_byte(moves, a, m);
    }
    return moves;
}

/* agent states in a plain array of four */
struct ArrayStore {
    SimpleSt* st;
    POM_HD SimpleSt load(int a) const { return st[a]; }
    POM_HD void store(int a, const SimpleSt& v) { st[a] = v; }
};

}
#endif
