/*
 * pom_core.cuh — one tick of one env on the packed record (pom_record.h).
 *
 * This is the body every kernel runs: the per-tick kernel on a record staged in shared memory,
 * the fused rollout kernel K times on a resident record.  One thread owns one env; the record
 * pointer `r` addresses shared memory on the device.  The four agents live in five packed
 * registers (`Agents`) for the whole tick; board, bomb ring and flame ring are read and written
 * in place.
 *
 * Semantics follow the reference tick exactly (src/bboard/step.cpp:9-284 and the helpers it
 * calls); each function cites the lines it re-states.  The reference's recursion
 * (SpawnFlame <-> SpawnFlameItem <-> ExplodeBombAt, bboard.cpp:24-57,111-118,198-263) is run
 * by an explicit stack of 32-bit frames (`explode`), its tail recursion
 * (AgentBombChainReversion, step_utility.cpp:62-128) by a loop (`revert_chain`).
 *
 * The header also compiles as plain C++ (POM_HD expands to `inline`); tests/hostsim builds it
 * that way to differential-test the tick logic on the CPU.  That build is test-only: the
 * product library contains device code only and has no CPU stepping path.
 */
#ifndef POM_CORE_CUH_
#define POM_CORE_CUH_

#include <stdint.h>
#include "pom_record.h"
#include "pom_state.h"

#if defined(__CUDACC__)
#define POM_HD __host__ __device__ inline
#define POM_HD_COLD __host__ __device__ __noinline__   /* rare paths: one out-of-line copy keeps the hot code small */
#define POM_LOOP _Pragma("unroll 1")   /* data-dependent trip counts: unrolling only bloats the code (I-cache) */
#else
#define POM_HD inline
#define POM_HD_COLD inline
#define POM_LOOP
#endif

namespace pomcore
{

/* flags returned by step(): same bits as oracle/pom_oracle.h POM_ORC_* */
enum {
    F_D1_UNREACHABLE = 0x01,
    F_D3_NULL_BOMB   = 0x02,
    F_D4_BOMB_OVF    = 0x04,
    F_FLAME_OVF      = 0x08,
    F_BAD_MOVE       = 0x10,
    F_LOOP_GUARD     = 0x20,   /* D5: AgentBombChainReversion would recurse forever (canonical: the chain stops) */
    F_RANGE          = 0x40,   /* device only: a field left what the packed record can carry (maxBombCount / bombStrength > 255) */
    F_INTERNAL       = 0x80,   /* device only: a guard of the explosion machine tripped (depth / iteration bound) */
    F_INVALID_MASK   = 0xFE,
    /* POM_STEP_CONTINUE_UNDEFINED: D3 and D5 have a canonical continuation (DESIGN §1) and do not stop the env */
    F_INVALID_MASK_CONTINUE = F_INVALID_MASK & ~(F_D3_NULL_BOMB | F_LOOP_GUARD)
};

/* the four agents, one byte per agent in each word */
struct Agents {
    uint32_t pos;    /* x | y<<4                     */
    uint32_t bcnt;   /* bombCount (signed byte)      */
    uint32_t amax;   /* maxBombCount                 */
    uint32_t astr;   /* bombStrength                 */
    uint32_t flg;    /* AF_CANKICK | AF_DEAD         */
    int      alive;  /* aliveAgents                  */
};

/* byte i of w / w with byte i replaced by v: one PRMT on the device (the index is usually dynamic) */
POM_HD uint32_t byte_of(uint32_t w, int i)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, 0x4440u + uint32_t(i));
#else
    return (w >> (8 * i)) & 0xFFu;
#endif
}
POM_HD uint32_t with_byte(uint32_t w, int i, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, v, 0x3210u + (uint32_t(4 - i) << (4 * i)));
#else
    const int s = 8 * i;
    return (w & ~(0xFFu << s)) | ((v & 0xFFu) << s);
#endif
}
/* (index + i) % 20 for the FixedQueue rings: multiply-high, shift, multiply-subtract - three instructions without a branch
 * at every one of the ~40 places the ring arithmetic is inlined (the three-way form "a < 20 ? a : a < 40 ? a - 20 : a % 20"
 * was 474 instructions of the step kernel's image, and the image size is felt: see k_step_ws) */
POM_HD uint32_t ring20(uint32_t a) { return a % 20u; }
POM_HD uint32_t ring_next(uint32_t slot) { return slot == 19u ? 0u : slot + 1u; }
/* byte-wise equality of the four bytes of w with the byte v: 0x80 in every byte that matches */
POM_HD uint32_t bytes_equal(uint32_t w, uint32_t v)
{
    const uint32_t x = w ^ (v * 0x01010101u);
    return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}

/* byte-wise equality of two words: 0x80 in every byte where a and b agree */
POM_HD uint32_t bytes_equal2(uint32_t a, uint32_t b)
{
    const uint32_t x = a ^ b;
    return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}
/* byte k of the result = byte (k + n) % 4 of w */
POM_HD uint32_t rot_bytes(uint32_t w, int n)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, n == 1 ? 0x0321u : (n == 2 ? 0x1032u : 0x2103u));
#else
    return (w >> (8 * n)) | (w << (32 - 8 * n));
#endif
}
/* 0x80-per-byte mask -> 0xFF-per-byte mask */
POM_HD uint32_t expand_mask(uint32_t m) { return (m >> 7) * 0xFFu; }

POM_HD uint32_t& bomb_slot(uint8_t* r, uint32_t slot) { return reinterpret_cast<uint32_t*>(r + R_BOMBS)[slot]; }
POM_HD uint32_t& bomb_at(uint8_t* r, uint32_t logical) { return bomb_slot(r, ring20(r[R_BINDEX] + logical)); }

/* positions: p = x | y<<4 (0..10 each).  "Biased" q = p + 0x11 keeps -1 and 11 representable. */
POM_HD int cell_of(uint32_t p) { return int(p & 15u) + 11 * int(p >> 4); }
POM_HD bool oob_biased(uint32_t q)
{
    const uint32_t x = q & 15u, y = (q >> 4) & 15u;
    return x == 0u || x == 12u || y == 0u || y == 12u;
}
/* DesiredPosition, step_utility.cpp:9-31: UP y-1, DOWN y+1, LEFT x-1, RIGHT x+1, anything else stays */
POM_HD int move_delta(uint32_t m)
{
    return (m - 1u < 4u) ? int(int8_t(0x01FF10F0u >> (8u * (m - 1u)))) : 0;
}

/* Item predicates on cell codes, bboard.hpp:73-109 */
POM_HD bool c_is_flame(uint32_t c)   { return (c & 0x80u) != 0u; }
POM_HD bool c_is_wood(uint32_t c)    { return c - 2u < 5u; }
POM_HD bool c_is_powerup(uint32_t c) { return c - 9u < 3u; }
POM_HD bool c_is_walkable(uint32_t c) { return c == 0u || c_is_powerup(c); }
POM_HD bool c_is_agent(uint32_t c)   { return c - 13u < 4u; }
POM_HD bool c_is_static(uint32_t c)  { return c - 1u < 6u || c_is_powerup(c); }

POM_HD bool ag_dead(const Agents& A, int i) { return (byte_of(A.flg, i) & AF_DEAD) != 0u; }

POM_HD void ag_kill(Agents& A, int i)                                 /* State::Kill, bboard.hpp:474-481 */
{
    if(!ag_dead(A, i))
    {
        A.flg |= uint32_t(AF_DEAD) << (8 * i);
        A.alive--;
    }
}

POM_HD int first_set_byte(uint32_t m)   /* m has bits only at positions 7/15/23/31; index of the lowest one, m != 0 */
{
    /* plain ALU ops: find-first-set (BREV + FLO) goes to the quarter-rate XU pipe, which this kernel keeps busy */
    const uint32_t l = m & (0u - m);
    return int(((l >> 15) & 1u) | ((l >> 22) & 2u) | ((l >> 31) * 3u));
}

POM_HD int get_agent(const Agents& A, uint32_t p)                    /* State::GetAgent, bboard.cpp:289-299 */
{
    /* first LIVE agent standing on p: byte-parallel compare, dead agents masked out (AF_DEAD = bit 1) */
    const uint32_t eq = bytes_equal(A.pos, p) & ~(A.flg << 6);
    return eq ? first_set_byte(eq) : -1;
}

POM_HD int bomb_index(uint8_t* r, uint32_t p)                        /* GetBombIndex / GetBomb / HasBomb, bboard.cpp:265-311 */
{
    const int n = r[R_BCOUNT];
    POM_LOOP
    for(int i = 0; i < n; i++)
    {
        if((bomb_at(r, i) & 0xFFu) == p) return i;
    }
    return -1;
}

POM_HD void bombs_remove_at(uint8_t* r, int at)                      /* FixedQueue::RemoveAt, bboard.hpp:151-160 */
{
    const int n = r[R_BCOUNT];
    const uint32_t bi = r[R_BINDEX];
    POM_LOOP
    for(int i = at + 1; i < n; i++)
    {
        const uint32_t t = ring20(bi + i);
        bomb_slot(r, (t + 19u) % 20u) = bomb_slot(r, t);
    }
    r[R_BCOUNT] = uint8_t(n - 1);
}

/* origin position of a flame cell code (FLAME_ID, bboard.hpp:98-101, through the slot indirection) */
POM_HD uint32_t flame_origin(const uint8_t* r, uint32_t c)
{
    const uint32_t slot = (c >> 2) & 31u;
    return slot == uint32_t(C_FLAME_ORPHAN_SLOT) ? 0u : r[R_FPOS + (slot % 20u)];
}

POM_HD void pop_flame(uint8_t* r)                                    /* State::PopFlame, bboard.cpp:148-180 */
{
    const uint32_t fi = r[R_FINDEX];
    const uint32_t p = r[R_FPOS + fi];
    int s = r[R_FSTR + fi];
    if(s > 10) s = 10;
    const int x = int(p & 15u), y = int(p >> 4);
    const uint32_t own = uint32_t(C_FLAME) | (fi << 2);   /* cells written by this very flame carry its slot */
    POM_LOOP
    for(int i = -s; i <= s; i++)
    {
        const int cx = x + i, cy = y + i;
        if(cx >= 0 && cx < 11)
        {
            uint8_t* cell = r + R_BOARD + cx + 11 * y;
            const uint32_t c = *cell;
            if(c_is_flame(c) && ((c & 0xFCu) == own || flame_origin(r, c) == p))
            {
                const uint32_t pw = c & 3u;                          /* FlagItem, bboard.cpp:182-189 */
                *cell = uint8_t(pw ? 8u + pw : 0u);
            }
        }
        if(cy >= 0 && cy < 11)
        {
            uint8_t* cell = r + R_BOARD + x + 11 * cy;
            const uint32_t c = *cell;
            if(c_is_flame(c) && ((c & 0xFCu) == own || flame_origin(r, c) == p))
            {
                const uint32_t pw = c & 3u;
                *cell = uint8_t(pw ? 8u + pw : 0u);
            }
        }
    }
    r[R_FINDEX] = uint8_t(ring20(fi + 1u));                          /* PopElem, bboard.hpp:131-137 */
    r[R_FCOUNT] = uint8_t(r[R_FCOUNT] - 1);
}

/* util::TickFlames, step_utility.cpp:208-222, in two halves so that kernels can run the (rare, long) pops
 * of a whole CTA tile with dense warps: flames_age() decrements every timer and says whether the front flame
 * expired; flames_pop_due() is the loop `for i < flameCount: if flames[0].timeLeft == 0 PopFlame()`. */
POM_HD bool flames_age(uint8_t* r)
{
    const int n = r[R_FCOUNT];
    if(n == 0) return false;
    uint32_t slot = r[R_FINDEX];
    POM_LOOP
    for(int i = 0; i < n; i++, slot = ring_next(slot))
    {
        uint8_t* t = r + R_FTIME + slot;
        *t = uint8_t(*t - 1);
    }
    /* a front flame whose timer is already negative never pops (in the reference either, Q10) and counts down for ever:
     * before the signed byte would wrap, the env leaves what the record can carry.  (pack() accepts timers in
     * [-16, 100], so no other entry can get near the limit while it waits for the front.) */
    const uint32_t front = r[R_FTIME + r[R_FINDEX]];
    if(front == 0x80u) r[R_STATUS] |= POM_STATUS_INVALID;
    return front == 0u;
}

POM_HD void flames_pop_due(uint8_t* r)
{
    const int n = r[R_FCOUNT];
    POM_LOOP
    for(int i = 0; i < n; i++)
    {
        if(r[R_FTIME + r[R_FINDEX]] == 0) pop_flame(r);
        else break;   /* flames[0] unchanged => no later iteration can pop either */
    }
}

POM_HD void tick_flames(uint8_t* r)
{
    if(flames_age(r)) flames_pop_due(r);
}

/*
 * Explosion machine: State::SpawnFlame (bboard.cpp:198-263) with SpawnFlameItem (:24-57) and the nested
 * State::ExplodeBombAt (:111-118) it triggers, depth-first in the reference's order (rays +x, -x, +y, -y).
 * One loop iteration handles one cell of one ray, so lanes that are in different rays, cells or nesting
 * depths still execute the same instructions.  Per spawn ("frame") the live state is: flame slot, ray d,
 * cells left in the ray, current cell index, and the logical index j of the bomb whose ExplodeBombAt opened
 * the frame (31 = a bare SpawnFlame: ExplodeTopBomb and fixtures, the caller does the epilogue).  A parent
 * frame is 32 bits on an explicit stack; the spawn's strength is read back from its flame-queue entry.
 * ExplodeBombAt's epilogue re-reads bombs[j] AFTER the nested explosions (SURVEY Q6).
 */
POM_HD_COLD void explode(uint8_t* r, Agents& A, uint32_t p0, uint32_t strength0, uint32_t j0, int& flags)
{
    uint32_t stack[24];
    int sp = 0;
    uint32_t slot = 0, d = 0, rem = 0, ci = 0, j = j0;
    uint32_t rooms = 0, ci0 = 0;                /* per spawn: cells to the border on the four rays, origin cell */
    int stride = 0;
    uint32_t p = p0, strength = strength0;
    bool start = true;
    POM_LOOP
    for(int guard = 0; guard < 8192; guard++)
    {
        if(start)
        {
            /* SpawnFlame prologue :200-218 */
            const uint32_t fc = r[R_FCOUNT];
            if(fc >= 20u) flags |= F_FLAME_OVF;
            slot = ring20(r[R_FINDEX] + fc);
            r[R_FPOS + slot] = uint8_t(p);
            r[R_FSTR + slot] = uint8_t(strength);
            r[R_FTIME + slot] = uint8_t(POM_FLAME_LIFETIME);
            r[R_FCOUNT] = uint8_t(fc + 1u);
            const uint32_t x = p & 15u, y = p >> 4;
            rooms = (10u - x) | (x << 8) | ((10u - y) << 16) | (y << 24);         /* ray bounds :223,234,245,256 */
            ci0 = x + 11u * y;
            const uint32_t c = r[R_BOARD + ci0];
            if(c_is_agent(c)) ag_kill(A, int(c) - C_AGENT0);
            r[R_BOARD + ci0] = uint8_t(C_FLAME | (slot << 2));
            d = 0xFFFFFFFFu;            /* the ray set-up below advances to ray 0 */
            rem = 0;
            start = false;
        }
        if(rem == 0u)
        {
            /* next ray of this spawn, or the spawn is complete */
            d++;
            if(d < 4u)
            {
                const uint32_t room = (rooms >> (8u * d)) & 0xFFu;
                rem = strength < room ? strength : room;
                stride = int(int8_t(0xF50BFF01u >> (8u * d)));            /* +1, -1, +11, -11 */
                ci = ci0;
                /* no `continue`: fall through to the first cell of the new ray in this very iteration, so that
                 * lanes which just finished a ray stay in step with lanes that are in the middle of one */
                if(rem == 0u) continue;
            }
            else
            {
            if(j != 31u)
            {
                /* ExplodeBombAt epilogue :116-117 */
                const uint32_t b = bomb_at(r, j);
                const int id = int((b >> 8) & 3u);
                A.bcnt = with_byte(A.bcnt, id, byte_of(A.bcnt, id) - 1u);
                bombs_remove_at(r, int(j));
            }
            if(sp == 0) return;
            /* back in the parent's SpawnFlameItem, after its ExplodeBombAt call (:42-52): the cell now holds
             * the child's flame (not RIGID, not wood), so it takes the parent's signature and the ray goes on */
            const uint32_t f = stack[--sp];
            slot = f & 31u; d = (f >> 5) & 3u; rem = (f >> 7) & 15u; ci = (f >> 11) & 127u; j = (f >> 18) & 31u;
            stride = int(int8_t(0xF50BFF01u >> (8u * d)));
            const uint32_t po = r[R_FPOS + slot];
            const uint32_t x = po & 15u, y = po >> 4;
            rooms = (10u - x) | (x << 8) | ((10u - y) << 16) | (y << 24);
            ci0 = x + 11u * y;
            strength = r[R_FSTR + slot];
            r[R_BOARD + ci] = uint8_t(C_FLAME | (slot << 2));
            continue;
            }
        }
        /* SpawnFlameItem on the next cell of the ray */
        ci = uint32_t(int(ci) + stride);
        rem--;
        uint8_t* cell = r + R_BOARD + ci;
        const uint32_t c = *cell;
        if(c == uint32_t(C_RIGID)) { rem = 0; continue; }                 /* :53-56 */
        if(c_is_wood(c))                                                  /* :45-51: only one wood per ray */
        {
            *cell = uint8_t(C_FLAME | (slot << 2) | ((c - 2u) & 3u));
            rem = 0;
            continue;
        }
        const bool isAgent = c_is_agent(c);
        if(isAgent || c == uint32_t(C_BOMB))                              /* :26-40 */
        {
            if(isAgent) ag_kill(A, int(c) - C_AGENT0);
            const uint32_t cp = (ci % 11u) | ((ci / 11u) << 4);
            const int jj = bomb_index(r, cp);
            if(jj >= 0)
            {
                if(sp >= 24) { flags |= F_INTERNAL; return; }
                stack[sp++] = slot | (d << 5) | (rem << 7) | (ci << 11) | (j << 18);
                const uint32_t b = bomb_at(r, jj);
                p = cp;
                strength = byte_of(A.astr, int((b >> 8) & 3u));           /* owner's CURRENT strength (Q5) */
                j = uint32_t(jj);
                start = true;
                continue;
            }
        }
        *cell = uint8_t(C_FLAME | (slot << 2));
    }
    flags |= F_INTERNAL;
}

/* util::AgentBombChainReversion, step_utility.cpp:62-128 (tail recursion -> loop).
 * bd[k] = biased destination of bomb k snapshotted before the pre-pass (step.cpp:191-192). */
POM_HD_COLD void revert_chain(uint8_t* r, Agents& A, uint32_t moves, const uint8_t* bd, int agentID, int& flags)
{
    POM_LOOP
    for(int guard = 0; guard < 64; guard++)
    {
        const uint32_t ap = byte_of(A.pos, agentID);
        const uint32_t oq = uint32_t(int(ap + 0x11u) - move_delta(byte_of(moves, agentID)));   /* OriginPosition :33-55 */
        if(oob_biased(oq)) return;
        const uint32_t origin = oq - 0x11u;
        const int indexOriginAgent = get_agent(A, origin);
        int bombDestIndex = -1;
        int n = r[R_BCOUNT];
        if(n > 20) n = 20;
        POM_LOOP
        for(int k = 0; k < n; k++)
        {
            if(bd[k] == oq) { bombDestIndex = k; break; }
        }
        A.pos = with_byte(A.pos, agentID, origin);
        r[R_BOARD + cell_of(origin)] = uint8_t(C_AGENT0 + agentID);
        /* D5: an agent whose move is IDLE/BOMB finds itself at its "origin": the reference recurses
         * forever here (hang at -O3, stack overflow at -O0); canonical = flag the env and stop */
        if(indexOriginAgent == agentID) { flags |= F_LOOP_GUARD; return; }
        if(indexOriginAgent != -1)
        {
            agentID = indexOriginAgent;
            continue;
        }
        if(bombDestIndex != -1)
        {
            uint32_t& b = bomb_at(r, bombDestIndex);
            const uint32_t bq = bd[bombDestIndex];
            const uint32_t obq = uint32_t(int(bq) - move_delta((b >> 20) & 15u));
            if(obq == bq)
            {
                /* bounced back onto a bomb he laid himself (:102-106) */
                r[R_BOARD + cell_of(obq - 0x11u)] = uint8_t(C_AGENT0 + agentID);
                return;
            }
            const uint32_t ob = obq - 0x11u;
            const int hasAgent = get_agent(A, ob);
            b = (b & ~0xF00000u);                                     /* SetBombDirection(IDLE) */
            b = (b & ~0xFFu) + ob;                                    /* SetBombPosition        */
            r[R_BOARD + cell_of(ob)] = uint8_t(C_BOMB);
            if(hasAgent != -1)
            {
                agentID = hasAgent;
                continue;
            }
        }
        return;
    }
    flags |= F_LOOP_GUARD;
}

POM_HD uint32_t bomb_dest_biased(uint32_t b)                         /* util::DesiredPosition(Bomb), step_utility.cpp:57-60 */
{
    return uint32_t(int((b & 0xFFu) + 0x11u) + move_delta((b >> 20) & 15u));
}

POM_HD bool has_bomb_collision(uint8_t* r, uint32_t b, int index)    /* step_utility.cpp:279-293 */
{
    const uint32_t t = bomb_dest_biased(b);
    const int n = r[R_BCOUNT];
    POM_LOOP
    for(int i = index; i < n; i++)
    {
        const uint32_t o = bomb_at(r, i);
        if(o != b && bomb_dest_biased(o) == t) return true;
    }
    return false;
}

POM_HD void resolve_bomb_collision(uint8_t* r, Agents& A, uint32_t moves, const uint8_t* bd, int index, int& flags) /* step_utility.cpp:295-329 */
{
    uint32_t& b = bomb_at(r, index);
    const uint32_t t = bomb_dest_biased(b);
    bool collided = false;
    const int n = r[R_BCOUNT];
    POM_LOOP
    for(int i = index; i < n; i++)
    {
        uint32_t& o = bomb_at(r, i);
        if(o != b && bomb_dest_biased(o) == t)
        {
            o = o & ~0xF00000u;
            collided = true;
        }
    }
    if(collided && ((b >> 20) & 15u) != 0u)
    {
        b = b & ~0xF00000u;
        const int a = get_agent(A, b & 0xFFu);
        const uint32_t m = a >= 0 ? byte_of(moves, a) : 0u;
        if(a >= 0 && m != uint32_t(POM_MOVE_IDLE) && m != uint32_t(POM_MOVE_BOMB))
        {
            revert_chain(r, A, moves, bd, a, flags);
            r[R_BOARD + cell_of(b & 0xFFu)] = uint8_t(C_BOMB);       /* b re-read: the chain may have moved it */
        }
    }
}

/* Per-tick scratch shared by the movement phase. */
struct TickCtx {
    uint32_t onBomb;        /* 0x80 in byte a: a bomb queue entry sits on agent a's cell (State::HasBomb of the
                               agent's start-of-tick cell; kept exact when bombs are planted this tick)            */
    uint32_t anyDir;        /* non-zero iff some bomb in the queue has a direction: start-of-tick directions, kicks
                               and stale direction bits inherited by bombs planted this tick (SURVEY Q4)           */
    uint32_t dstBomb;       /* 0x80 in byte a: a start-of-tick bomb queue entry sits on agent a's DESTINATION      */
    uint32_t needRevert;    /* non-zero iff an agent may stand on a queue entry's cell after moving there this
                               tick: only then can the bomb pre-pass (step.cpp:195-227) bounce anyone back         */
};

/* leave the cell an agent stood on: BOMB if a queue entry sits there, else PASSAGE (step.cpp:89-96,127-134) */
POM_HD void vacate(uint8_t* r, uint32_t p, const TickCtx& T, int i)
{
    r[R_BOARD + cell_of(p)] = uint8_t(((T.onBomb >> (8 * i + 7)) & 1u) ? C_BOMB : C_PASSAGE);
}

/* body of the movement loop for agent i, step.cpp:46-184 */
POM_HD void move_agent(uint8_t* r, Agents& A, TickCtx& T, uint32_t moves, uint32_t dq, bool ouroboros, int i, int& flags)
{
    const uint32_t m = byte_of(moves, i);
    if(ag_dead(A, i) || m == uint32_t(POM_MOVE_IDLE)) return;
    const uint32_t p = byte_of(A.pos, i);
    if(m == uint32_t(POM_MOVE_BOMB))
    {
        /* PlantBombModifiedLife(x, y, i, BOMB_LIFETIME + 1), bboard.cpp:125-146; the slot's stale
         * direction / moved bits survive (Q4); ticked to 10 at the end of this Step (Q3) */
        if(int(int8_t(byte_of(A.bcnt, i))) >= int(byte_of(A.amax, i))) return;
        const uint32_t cnt = r[R_BCOUNT];
        if(cnt >= 20u) flags |= F_D4_BOMB_OVF;
        uint32_t& b = bomb_slot(r, ring20(r[R_BINDEX] + cnt));
        b = (b & ~0xF00u) + (uint32_t(i) << 8);
        b = (b & ~0xFFu) + p;
        b = (b & ~0xF000u) + (byte_of(A.astr, i) << 12);
        b = (b & ~0xF0000u) + (uint32_t(POM_BOMB_LIFETIME + 1) << 16);
        A.bcnt = with_byte(A.bcnt, i, byte_of(A.bcnt, i) + 1u);
        r[R_BCOUNT] = uint8_t(cnt + 1u);
        T.onBomb |= bytes_equal(A.pos, p);
        T.anyDir |= b & 0xF00000u;
        return;
    }
    const uint32_t d = byte_of(dq, i);
    if(oob_biased(d)) return;                                        /* :63 */
    const uint32_t dp = d - 0x11u;
    uint8_t* dcell = r + R_BOARD + cell_of(dp);
    uint8_t* ocell = r + R_BOARD + cell_of(p);
    uint32_t item = *dcell;
    if(ouroboros && bomb_index(r, dp) >= 0) item = C_BOMB;           /* :71-82 */
    if(c_is_flame(item))                                             /* :84-99 */
    {
        ag_kill(A, i);
        if(*ocell == uint32_t(C_AGENT0 + i)) vacate(r, p, T, i);
        return;
    }
    /* HasDPCollision, step_utility.cpp:264-277: another LIVE agent with the same destination */
    if(bytes_equal(dq, d) & ~(A.flg << 6) & ~(0x80u << (8 * i))) return;
    if(c_is_powerup(item))                                           /* ConsumePowerup, step_utility.cpp:247-262 */
    {
        /* the reference counts these up in ints without bound; the record holds bytes */
        if(item == uint32_t(C_EXTRABOMB)) { if(byte_of(A.amax, i) == 255u) flags |= F_RANGE; A.amax = with_byte(A.amax, i, byte_of(A.amax, i) + 1u); }
        else if(item == uint32_t(C_INCRRANGE)) { if(byte_of(A.astr, i) == 255u) flags |= F_RANGE; A.astr = with_byte(A.astr, i, byte_of(A.astr, i) + 1u); }
        else A.flg |= uint32_t(AF_CANKICK) << (8 * i);
        item = C_PASSAGE;
    }
    if(item == uint32_t(C_PASSAGE) || (ouroboros && c_is_agent(item)))   /* :120-140 */
    {
        if(*ocell == uint32_t(C_AGENT0 + i)) vacate(r, p, T, i);
        *dcell = uint8_t(C_AGENT0 + i);
        A.pos = with_byte(A.pos, i, dp);
    }
    else if(item == uint32_t(C_BOMB))                                /* :147-184: kick, or step onto the bomb (Q2) */
    {
        vacate(r, p, T, i);
        *dcell = uint8_t(C_AGENT0 + i);
        A.pos = with_byte(A.pos, i, dp);
        if(byte_of(A.flg, i) & AF_CANKICK)
        {
            const int bi = bomb_index(r, dp);
            if(bi < 0) flags |= F_D3_NULL_BOMB;                      /* the reference dereferences nullptr here (D3) */
            else
            {
                uint32_t& b = bomb_at(r, bi);
                b = (b & ~0xF00000u) + (m << 20);
                T.anyDir |= b & 0xF00000u;
            }
        }
    }
}

POM_HD int popcount32(uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}

/*
 * The movement loop of Step (step.cpp:39-185) for all four agents at once, one byte per agent.
 *
 * Applies when the order of the loop cannot matter: no two agents would swap cells (FixSwitchMove,
 * step_utility.cpp:154-170, leaves every destination alone), no live agent wants the cell of another live
 * agent (ResolveDependencies, :172-205: every agent is a root, the loop runs 0,1,2,3), and the board shows
 * every live agent on its cell (so live agents stand on four different cells).  Then agent i reads only its
 * destination cell and writes only its own and its destination cell; two live agents with the same
 * destination both stop at HasDPCollision (:264-277) before writing anything - or both burn; the bomb ring
 * is appended to in agent order.  In the bench workload 99.9 % of the env-ticks qualify; with 32 envs per warp
 * the serial loop below is still entered by 2 % of the warps.
 * Returns false, having written NOTHING, when the tick does not qualify.
 */
POM_HD bool move_agents_fast(uint8_t* r, Agents& A, TickCtx& T, uint32_t moves, uint32_t dq, uint32_t posq, int& flags)
{
    const uint32_t H = 0x80808080u;
    const uint32_t live = ~(A.flg << 6) & H;
    const uint32_t l1 = rot_bytes(live, 1), l2 = rot_bytes(live, 2), l3 = rot_bytes(live, 3);
    /* e_k, byte a: the destination of agent a is the cell of agent (a + k) % 4 */
    const uint32_t e1 = bytes_equal2(dq, rot_bytes(posq, 1));
    const uint32_t e2 = bytes_equal2(dq, rot_bytes(posq, 2));
    const uint32_t e3 = bytes_equal2(dq, rot_bytes(posq, 3));
    const uint32_t swaps = (e1 & rot_bytes(e3, 1)) | (e2 & rot_bytes(e2, 2)) | (e3 & rot_bytes(e1, 3));   /* dead agents count (Q1) */
    const uint32_t deps = ((e1 & l1) | (e2 & l2) | (e3 & l3)) & live;
    if(swaps | deps) return false;

    const uint32_t isIdle = bytes_equal(moves, uint32_t(POM_MOVE_IDLE)), isBomb = bytes_equal(moves, uint32_t(POM_MOVE_BOMB));
    const uint32_t xs = dq & 0x0F0F0F0Fu, ys = (dq >> 4) & 0x0F0F0F0Fu;                  /* biased: on the board = 1..11 */
    const uint32_t oob = (~(xs + 0x7F7F7F7Fu) | (xs + 0x74747474u) | ~(ys + 0x7F7F7F7Fu) | (ys + 0x74747474u)) & H;
    const uint32_t mv = live & ~(isIdle | isBomb | oob);                                  /* agents that try to enter a cell (:63) */
    const uint32_t mvE = expand_mask(mv);
    const uint32_t tq = (dq & mvE) | (posq & ~mvE);                                       /* the others: their own cell, a safe address */
    const uint32_t dci = (tq & 0x0F0F0F0Fu) + ((tq >> 4) & 0x0F0F0F0Fu) * 11u - 0x0C0C0C0Cu;
    const uint32_t oci = (posq & 0x0F0F0F0Fu) + ((posq >> 4) & 0x0F0F0F0Fu) * 11u - 0x0C0C0C0Cu;
    uint8_t* bd = r + R_BOARD;
    const uint32_t items = uint32_t(bd[byte_of(dci, 0)]) | (uint32_t(bd[byte_of(dci, 1)]) << 8) |
                           (uint32_t(bd[byte_of(dci, 2)]) << 16) | (uint32_t(bd[byte_of(dci, 3)]) << 24);
    const uint32_t own = uint32_t(bd[byte_of(oci, 0)]) | (uint32_t(bd[byte_of(oci, 1)]) << 8) |
                         (uint32_t(bd[byte_of(oci, 2)]) << 16) | (uint32_t(bd[byte_of(oci, 3)]) << 24);
    if(~bytes_equal2(own, 0x100F0E0Du) & live) return false;      /* C_AGENT0 + a in byte a: fixtures and uploaded states may differ */

    const uint32_t flame = items & H;
    const uint32_t lo = items & 0x7F7F7F7Fu;
    const uint32_t passage = ~((lo + 0x7F7F7F7Fu) | items) & H;
    const uint32_t pwr = (lo + 0x77777777u) & ~(lo + 0x74747474u) & ~items & H;          /* 9..11 */
    const uint32_t bombc = bytes_equal(items, uint32_t(C_BOMB));
    const uint32_t c1 = bytes_equal2(dq, rot_bytes(dq, 1)), c2 = bytes_equal2(dq, rot_bytes(dq, 2));
    const uint32_t coll = (c1 & l1) | (c2 & l2) | (rot_bytes(c1, 3) & l3);               /* HasDPCollision */
    const uint32_t die = mv & flame;                                                      /* :84-99 */
    uint32_t go = mv & ~flame & ~coll & (passage | pwr | bombc);                          /* :101-184 */

    uint32_t pl = isBomb & live;                                                          /* PlantBombModifiedLife, as in move_agent */
    POM_LOOP
    while(pl)
    {
        const int a = first_set_byte(pl);
        pl &= pl - 1u;
        if(int(int8_t(byte_of(A.bcnt, a))) >= int(byte_of(A.amax, a))) continue;
        const uint32_t cnt = r[R_BCOUNT];
        if(cnt >= 20u) flags |= F_D4_BOMB_OVF;
        uint32_t& b = bomb_slot(r, ring20(r[R_BINDEX] + cnt));
        b = (b & ~0xF00u) + (uint32_t(a) << 8);
        b = (b & ~0xFFu) + byte_of(A.pos, a);
        b = (b & ~0xF000u) + (byte_of(A.astr, a) << 12);
        b = (b & ~0xF0000u) + (uint32_t(POM_BOMB_LIFETIME + 1) << 16);
        A.bcnt = with_byte(A.bcnt, a, byte_of(A.bcnt, a) + 1u);
        r[R_BCOUNT] = uint8_t(cnt + 1u);
        T.onBomb |= 0x80u << (8 * a);
        T.anyDir |= b & 0xF00000u;
    }
    uint32_t kick = go & bombc & (A.flg << 7);                                            /* :147-184 with canKick */
    /* Q2: an agent that cannot kick still steps onto the bomb and is bounced back by the bomb pre-pass
     * (step.cpp:170-184,195-227).  When no bomb has or gets a direction this tick, that round trip changes nothing: the
     * agent's cell and the bomb's cell end as they started, no one else reads either cell in between (no other live agent
     * has this agent's old cell or its destination as destination).  So such an agent simply stays.  With a direction
     * somewhere the general bomb phase may see the agent on the bomb: then it does step there. */
    if((T.anyDir | kick) == 0u) go &= ~(bombc & T.dstBomb);
    T.needRevert = go & T.dstBomb;

    const uint32_t vac = die | go;
    const uint32_t vacv = (T.onBomb >> 7) * uint32_t(C_BOMB);                             /* vacate(): BOMB or PASSAGE */
#if defined(__CUDACC__)
#pragma unroll
#endif
    for(int a = 0; a < 4; a++)
    {
        if(vac & (0x80u << (8 * a))) bd[byte_of(oci, a)] = uint8_t(byte_of(vacv, a));
        if(go & (0x80u << (8 * a))) bd[byte_of(dci, a)] = uint8_t(C_AGENT0 + a);
    }
    const uint32_t goE = expand_mask(go);
    A.pos = (A.pos & ~goE) | ((tq - 0x11111111u) & goE);
    const uint32_t pick = go & pwr;                                                       /* ConsumePowerup, step_utility.cpp:247-262 */
    if(pick)
    {
        const uint32_t b1 = (items << 6) & H, b0 = (items << 7) & H;                     /* 9 = 1001b, 10 = 1010b, 11 = 1011b */
        const uint32_t eb = pick & ~b1, ir = pick & b1 & ~b0, kk = pick & b1 & b0;
        if((bytes_equal(A.amax, 0xFFu) & eb) | (bytes_equal(A.astr, 0xFFu) & ir)) flags |= F_RANGE;
        A.amax = ((A.amax & 0x7F7F7F7Fu) + (eb >> 7)) ^ (A.amax & H);
        A.astr = ((A.astr & 0x7F7F7F7Fu) + (ir >> 7)) ^ (A.astr & H);
        A.flg |= kk >> 7;                                                                  /* AF_CANKICK */
    }
    POM_LOOP
    while(kick)
    {
        const int a = first_set_byte(kick);
        kick &= kick - 1u;
        const int bi = bomb_index(r, byte_of(tq, a) - 0x11u);
        if(bi < 0) flags |= F_D3_NULL_BOMB;
        else
        {
            uint32_t& b = bomb_at(r, bi);
            b = (b & ~0xF00000u) + (byte_of(moves, a) << 20);
            T.anyDir |= b & 0xF00000u;
        }
    }
    if(die)
    {
        A.flg |= die >> 6;                                                                 /* AF_DEAD */
        A.alive -= popcount32(die);
    }
    return true;
}

POM_HD void load_agents(const uint8_t* r, Agents& A)
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(r + R_APOS);
    A.pos = w[0]; A.bcnt = w[1]; A.amax = w[2]; A.astr = w[3]; A.flg = w[4];
    A.alive = int(int8_t(r[R_ALIVE]));
}

POM_HD void store_agents(uint8_t* r, const Agents& A)
{
    uint32_t* w = reinterpret_cast<uint32_t*>(r + R_APOS);
    w[0] = A.pos; w[1] = A.bcnt; w[2] = A.amax; w[3] = A.astr; w[4] = A.flg;
    r[R_ALIVE] = uint8_t(A.alive);
}

/* util::AgentBombChainReversion when EVERY bomb is idle (direction 0): destBombs[k] is then bomb k's own
 * cell, the bomb branch (step_utility.cpp:94-106) only re-writes the agent's cell, and the chain reduces to
 * walking agents back along their moves. */
POM_HD void revert_chain_idle(uint8_t* r, Agents& A, uint32_t moves, int agentID, int& flags)
{
    POM_LOOP
    for(int guard = 0; guard < 64; guard++)
    {
        const uint32_t ap = byte_of(A.pos, agentID);
        const uint32_t oq = uint32_t(int(ap + 0x11u) - move_delta(byte_of(moves, agentID)));
        if(oob_biased(oq)) return;
        const uint32_t origin = oq - 0x11u;
        const int indexOriginAgent = get_agent(A, origin);
        A.pos = with_byte(A.pos, agentID, origin);
        r[R_BOARD + cell_of(origin)] = uint8_t(C_AGENT0 + agentID);
        if(indexOriginAgent == agentID) { flags |= F_LOOP_GUARD; return; }    /* D5 */
        if(indexOriginAgent == -1) return;
        agentID = indexOriginAgent;
    }
    flags |= F_LOOP_GUARD;
}

/* The bomb phase of Step (step.cpp:187-278) in its general form: some bomb has a direction.  Rare
 * (needs a kick or a stale-direction plant), so it is kept out of line; the agents travel through the
 * record instead of registers. */
POM_HD_COLD int bomb_phase_general(uint8_t* r, uint32_t moves, uint32_t oldPos, int bc)
{
    int flags = 0;
    Agents A;
    load_agents(r, A);
    if(bc > 20) flags |= F_D4_BOMB_OVF;
    uint8_t bd[20];
    POM_LOOP
    for(int k = 0; k < bc && k < 20; k++) bd[k] = uint8_t(bomb_dest_biased(bomb_at(r, k)));   /* FillBombDestPos :191-192 */

    POM_LOOP
    for(int k = 0; k < bc; k++)                                      /* :195-227 */
    {
        uint32_t& b = bomb_at(r, k);
        const uint32_t bp = b & 0xFFu;
        const uint32_t t = bomb_dest_biased(b);
        bool blocked = oob_biased(t);
        if(!blocked)
        {
            const uint32_t c = r[R_BOARD + cell_of(t - 0x11u)];
            blocked = c_is_static(c) || c_is_agent(c);
        }
        if(blocked)
        {
            b = b & ~0xF00000u;
            const int a = get_agent(A, bp);
            if(a >= 0)
            {
                const uint32_t m = byte_of(moves, a);
                if(m != uint32_t(POM_MOVE_IDLE) && m != uint32_t(POM_MOVE_BOMB) &&
                        byte_of(A.pos, a) != byte_of(oldPos, a))
                {
                    revert_chain(r, A, moves, bd, a, flags);
                    if(get_agent(A, bp) == -1) r[R_BOARD + cell_of(bp)] = uint8_t(C_BOMB);
                }
            }
        }
    }

    for(int k = 0; k < int(r[R_BCOUNT]); k++)                        /* :230-278; the ring may shrink inside (Q7) */
    {
        uint32_t& b = bomb_at(r, k);
        if(((b >> 20) & 15u) == 0u && has_bomb_collision(r, b, k))
        {
            resolve_bomb_collision(r, A, moves, bd, k, flags);
            continue;
        }
        const uint32_t bp = b & 0xFFu;
        const uint32_t t = bomb_dest_biased(b);
        bool free_target = !oob_biased(t);
        uint8_t* tcell = r;
        if(free_target)
        {
            tcell = r + R_BOARD + cell_of(t - 0x11u);
            free_target = !c_is_static(*tcell);
        }
        if(free_target)
        {
            if(has_bomb_collision(r, b, k))
            {
                resolve_bomb_collision(r, A, moves, bd, k, flags);
                continue;
            }
            const uint32_t tp = t - 0x11u;
            b = (b & ~0xFFu) + tp;                                   /* SetBombPosition */
            uint8_t* ocell = r + R_BOARD + cell_of(bp);
            if(*ocell == uint32_t(C_BOMB) && bomb_index(r, bp) < 0) *ocell = uint8_t(C_PASSAGE);
            const uint32_t ti = *tcell;
            if(c_is_walkable(ti)) *tcell = uint8_t(C_BOMB);
            else if(c_is_flame(ti))
            {
                const int idx = bomb_index(r, tp);                   /* ExplodeBombAt(GetBombIndex(target)) :271 */
                const uint32_t eb = bomb_at(r, idx);
                explode(r, A, tp, byte_of(A.astr, int((eb >> 8) & 3u)), uint32_t(idx), flags);
            }
        }
        else
        {
            b = b & ~0xF00000u;
        }
    }
    store_agents(r, A);
    return flags;
}

/* State::ExplodeBombAt(idx) (bboard.cpp:111-118) out of line, agents through the record */
POM_HD_COLD int explode_bomb_at_cold(uint8_t* r, uint32_t p, int idx)
{
    int flags = 0;
    Agents A;
    load_agents(r, A);
    const uint32_t eb = bomb_at(r, idx);
    explode(r, A, p, byte_of(A.astr, int((eb >> 8) & 3u)), uint32_t(idx), flags);
    store_agents(r, A);
    return flags;
}

/* The move loop of Step (:230-278) when every bomb is idle: a bomb whose cell reads PASSAGE is re-stamped
 * BOMB, a bomb whose cell reads FLAMES explodes — unless a later ring entry with a different value sits on
 * the same cell (HasBombCollision -> `continue`, Q13). */
POM_HD void bomb_move_idle(uint8_t* r, Agents& A, int& flags)
{
    POM_LOOP
    for(int k = 0; k < int(r[R_BCOUNT]); k++)
    {
        const uint32_t b = bomb_at(r, k);
        const uint32_t bp = b & 0xFFu;
        uint8_t* cell = r + R_BOARD + cell_of(bp);
        const uint32_t c = *cell;
        if(c == uint32_t(C_PASSAGE) || c_is_flame(c))
        {
            bool collides = false;
            const int n = r[R_BCOUNT];
            POM_LOOP
            for(int i = k + 1; i < n; i++)
            {
                const uint32_t o = bomb_at(r, i);
                if(o != b && (o & 0xFFu) == bp) { collides = true; break; }
            }
            if(collides) continue;
            if(c == uint32_t(C_PASSAGE)) *cell = uint8_t(C_BOMB);
            else
            {
                store_agents(r, A);
                flags |= explode_bomb_at_cold(r, bp, bomb_index(r, bp));
                load_agents(r, A);
            }
        }
    }
}

/* bboard::Step, step.cpp:9-284, is split in four pieces so that the kernels can run the two rare, long,
 * divergent pieces (flame pops at the start, timed-out bomb explosions at the end) for a whole CTA tile
 * with dense warps:   flames_age -> [flames_pop_due] -> step_body -> [step_explode_due]
 * step_body is everything between TickFlames and the explosion loop of TickBombs; it returns the F_* flags
 * and sets `explode_due` when bombs[0] has timed out.  `moves`: byte a = Move of agent a. */
POM_HD int step_body(uint8_t* r, uint32_t moves, bool& explode_due, bool explode_inline = false)
{
    int flags = 0;
    explode_due = false;
    /* a move byte outside 0..5 is treated as IDLE and flagged (all four bytes tested at once) */
    if((((moves & 0x7F7F7F7Fu) + 0x7A7A7A7Au) | moves) & 0x80808080u)
    {
        for(int a = 0; a < 4; a++)
        {
            if(byte_of(moves, a) > 5u) { moves = with_byte(moves, a, 0u); flags |= F_BAD_MOVE; }
        }
    }

    Agents A;
    load_agents(r, A);
    const uint32_t oldPos = A.pos;                                   /* FillPositions :24 */
    const uint32_t posq = A.pos + 0x11111111u;

    /* destinations, one biased byte per agent (kept in a register: a dynamically indexed array would
     * live in local memory) */
    uint32_t dq = 0u;
    for(int a = 0; a < 4; a++)                                       /* FillDestPos :25 */
        dq |= (uint32_t(int(byte_of(posq, a)) + move_delta(byte_of(moves, a))) & 0xFFu) << (8 * a);

    /* which agents stand on a bomb queue entry (State::HasBomb of their cell, used when they leave it), and which
     * are heading for one */
    TickCtx T;
    T.onBomb = 0u;
    T.anyDir = 0u;
    T.dstBomb = 0u;
    {
        const int bc0 = r[R_BCOUNT];
        uint32_t slot = r[R_BINDEX];
        POM_LOOP
        for(int k = 0; k < bc0; k++, slot = ring_next(slot))
        {
            const uint32_t b = bomb_slot(r, slot);
            const uint32_t bq = ((b & 0xFFu) + 0x11u) * 0x01010101u;
            T.onBomb |= bytes_equal2(posq, bq);
            T.dstBomb |= bytes_equal2(dq, bq);
            T.anyDir |= b & 0xF00000u;
        }
    }
    if(!move_agents_fast(r, A, T, moves, dq, posq, flags))
    {
    /* tgt[a]: 0x80 in byte b iff agent a's destination is agent b's cell.  The same four masks serve
     * FixSwitchMove (:26, step_utility.cpp:154-170; dead agents NOT skipped, Q1) and ResolveDependencies
     * (:32, step_utility.cpp:172-205). */
    uint32_t tgt[4];
#pragma unroll
    for(int a = 0; a < 4; a++) tgt[a] = bytes_equal(posq, byte_of(dq, a));
#pragma unroll
    for(int a = 0; a < 4; a++)
    {
#pragma unroll
        for(int b = a + 1; b < 4; b++)
        {
            if((tgt[a] & (0x80u << (8 * b))) && (tgt[b] & (0x80u << (8 * a))))
            {
                /* a and b would swap cells: both stay (rare, so the masks are simply recomputed) */
                dq = with_byte(dq, a, byte_of(posq, a));
                dq = with_byte(dq, b, byte_of(posq, b));
                tgt[a] = bytes_equal(posq, byte_of(posq, a));
                tgt[b] = bytes_equal(posq, byte_of(posq, b));
            }
        }
    }

    uint32_t dep = 0xFFFFFFFFu, roots = 0xFFFFFFFFu;
    int rootNumber = 0;
    const uint32_t liveMask = ~(A.flg << 6);
#pragma unroll
    for(int a = 0; a < 4; a++)
    {
        bool isRoot = true;
        if(!ag_dead(A, a))
        {
            /* first other LIVE agent standing on a's destination */
            const uint32_t hit = tgt[a] & liveMask & ~(0x80u << (8 * a));
            if(hit)
            {
                dep = with_byte(dep, first_set_byte(hit), uint32_t(a));
                isRoot = false;
            }
        }
        if(isRoot) roots = with_byte(roots, rootNumber++, uint32_t(a));
    }
    const bool ouroboros = rootNumber == 0;

    {
        int rootIdx = 0;
        uint32_t i = rootNumber == 0 ? 0u : byte_of(roots, 0);
        for(int k = 0; k < 4; k++)                                   /* :39-185 */
        {
            if(i == 0xFFu)
            {
                rootIdx++;
                /* D1: the reference indexes roots/moves/agents with -1 here; canonical = stop */
                if(rootIdx > 3 || byte_of(roots, rootIdx) == 0xFFu) { flags |= F_D1_UNREACHABLE; break; }
                i = byte_of(roots, rootIdx);
            }
            move_agent(r, A, T, moves, dq, ouroboros, int(i), flags);
            i = byte_of(dep, int(i));
        }
    }
    T.needRevert = A.pos ^ oldPos;
    }

    int bc = r[R_BCOUNT];
    if(bc > 0)
    {
        bool timers_ticked = false;
        if(T.anyDir)
        {
            /* some bomb moves (a kick, or a stale-direction plant): the general form of :187-278, out of line */
            uint32_t slot = r[R_BINDEX];
            POM_LOOP
            for(int k = 0; k < bc; k++, slot = ring_next(slot)) bomb_slot(r, slot) &= ~0xF000000u;   /* ResetBombFlags :188 */
            store_agents(r, A);
            flags |= bomb_phase_general(r, moves, oldPos, bc);
            load_agents(r, A);
        }
        else
        {
            /* Every bomb is idle.  One pass does ResetBombFlags (:188) and the idle form of the pre-pass (:195-227:
             * bounce back an agent that walked onto a bomb this tick), and notes whether the idle form of the move
             * loop (:230-278) has anything to do: it only re-stamps / explodes bombs whose cell reads PASSAGE / FLAMES.
             * Reversions write AGENT or BOMB codes only, so they cannot create such a cell behind the pass. */
            bool needMove = false;
            const bool anyAgentMoved = T.needRevert != 0u;
            uint32_t slot = r[R_BINDEX];
            POM_LOOP
            for(int k = 0; k < bc; k++, slot = ring_next(slot))
            {
                const uint32_t b = bomb_slot(r, slot);
                /* ResetBombFlags, and — speculatively — ReduceBombTimer of TickBombs (:283): in the common tick
                 * nothing between here and TickBombs touches the ring, so the timers are ticked in this pass */
                bomb_slot(r, slot) = (b & ~0xF000000u) - (1u << 16);
                const uint32_t bp = b & 0xFFu;
                const uint32_t c = r[R_BOARD + cell_of(bp)];
                needMove = needMove || c == uint32_t(C_PASSAGE) || c_is_flame(c);
                if(anyAgentMoved && (c_is_agent(c) || c_is_static(c)))
                {
                    const int a = get_agent(A, bp);
                    if(a >= 0)
                    {
                        const uint32_t m = byte_of(moves, a);
                        if(m != uint32_t(POM_MOVE_IDLE) && m != uint32_t(POM_MOVE_BOMB) &&
                                byte_of(A.pos, a) != byte_of(oldPos, a))
                        {
                            revert_chain_idle(r, A, moves, a, flags);
                            if(get_agent(A, bp) == -1) r[R_BOARD + cell_of(bp)] = uint8_t(C_BOMB);
                        }
                    }
                }
            }
            timers_ticked = true;
            if(needMove)
            {
                /* rare: the move loop may explode bombs (RemoveAt leaves un-ticked stale copies in the reference),
                 * so take the speculative tick back, run the loop, and let TickBombs tick as usual */
                slot = r[R_BINDEX];
                POM_LOOP
                for(int k = 0; k < bc; k++, slot = ring_next(slot)) bomb_slot(r, slot) += (1u << 16);
                timers_ticked = false;
                bomb_move_idle(r, A, flags);
            }
        }

        /* util::TickBombs :283, step_utility.cpp:224-245 */
        bc = r[R_BCOUNT];
        if(!timers_ticked)
        {
            uint32_t slot = r[R_BINDEX];
            POM_LOOP
            for(int k = 0; k < bc; k++, slot = ring_next(slot)) bomb_slot(r, slot) -= (1u << 16);   /* ReduceBombTimer, bboard.hpp:308-311 */
        }
        explode_due = bc > 0 && ((bomb_slot(r, r[R_BINDEX]) >> 16) & 15u) == 0u;
        if(explode_due && explode_inline)
        {
            /* the explosion loop of util::TickBombs with the agents still in registers (see step_explode_due) */
            POM_LOOP
            for(int k = 0; k < bc && r[R_BCOUNT] > 0; k++)
            {
                const uint32_t c = bomb_slot(r, r[R_BINDEX]);
                if(((c >> 16) & 15u) != 0u) break;
                explode(r, A, c & 0xFFu, (c >> 12) & 15u, 31u, flags);
                const int id = int((bomb_slot(r, r[R_BINDEX]) >> 8) & 3u);
                A.bcnt = with_byte(A.bcnt, id, byte_of(A.bcnt, id) - 1u);
                r[R_BINDEX] = uint8_t(ring_next(r[R_BINDEX]));
                r[R_BCOUNT] = uint8_t(r[R_BCOUNT] - 1);
            }
            explode_due = false;
        }
    }

    store_agents(r, A);
    return flags;
}

/* the explosion loop of util::TickBombs (step_utility.cpp:231-244): while bombs[0] has timed out,
 * ExplodeTopBomb (bboard.cpp:191-196, strength stored in the bomb) and PopBomb (:93-97). */
POM_HD int step_explode_due(uint8_t* r)
{
    int flags = 0;
    Agents A;
    load_agents(r, A);
    const int bc = r[R_BCOUNT];
    POM_LOOP
    for(int k = 0; k < bc && r[R_BCOUNT] > 0; k++)
    {
        const uint32_t c = bomb_slot(r, r[R_BINDEX]);
        if(((c >> 16) & 15u) != 0u) break;
        explode(r, A, c & 0xFFu, (c >> 12) & 15u, 31u, flags);
        const int id = int((bomb_slot(r, r[R_BINDEX]) >> 8) & 3u);
        A.bcnt = with_byte(A.bcnt, id, byte_of(A.bcnt, id) - 1u);
        r[R_BINDEX] = uint8_t(ring_next(r[R_BINDEX]));
        r[R_BCOUNT] = uint8_t(r[R_BCOUNT] - 1);
    }
    store_agents(r, A);
    return flags;
}

/* ray d of a spawn at p (order +x, -x, +y, -y, :220-262): cells up to the border or `strength`; sets the cell stride */
POM_HD uint32_t ray_length(uint32_t p, uint32_t strength, uint32_t d, int& stride)
{
    const uint32_t x = p & 15u, y = p >> 4;
    const uint32_t rooms = (10u - x) | (x << 8) | ((10u - y) << 16) | (y << 24);
    const uint32_t room = (rooms >> (8u * d)) & 0xFFu;
    stride = int(int8_t(0xF50BFF01u >> (8u * d)));                    /* +1, -1, +11, -11 */
    return strength < room ? strength : room;
}

/* ---------------------------------------------------------------------------------------------
 * Arm-parallel form of State::PopFlame (bboard.cpp:148-180) for the warp-cooperative tick (warp_pop_due): the cross of
 * +-strength cells is four arms and a centre; every cell is cleared from its own old value and the (unchanged) flame
 * positions alone, so the arms need no order.  The ring is popped after all arms are done.
 * ------------------------------------------------------------------------------------------- */
POM_HD void pop_flame_cell(uint8_t* r, uint32_t ci, uint32_t own, uint32_t p)
{
    uint8_t* cell = r + R_BOARD + ci;
    const uint32_t c = *cell;
    if(c_is_flame(c) && ((c & 0xFCu) == own || flame_origin(r, c) == p))
    {
        const uint32_t pw = c & 3u;                                   /* FlagItem, bboard.cpp:182-189 */
        *cell = uint8_t(pw ? 8u + pw : 0u);
    }
}

/* arm d (+x, -x, +y, -y) of the front flame's cross; d == 0 also clears the centre */
POM_HD void pop_flame_arm(uint8_t* r, uint32_t d)
{
    const uint32_t fi = r[R_FINDEX];
    const uint32_t p = r[R_FPOS + fi];
    uint32_t s = r[R_FSTR + fi];
    if(s > 10u) s = 10u;
    const uint32_t own = uint32_t(C_FLAME) | (fi << 2);
    int stride;
    const uint32_t len = ray_length(p, s, d, stride);
    uint32_t ci = uint32_t(cell_of(p));
    if(d == 0u) pop_flame_cell(r, ci, own, p);
    POM_LOOP
    for(uint32_t k = 0; k < len; k++)
    {
        ci = uint32_t(int(ci) + stride);
        pop_flame_cell(r, ci, own, p);
    }
}

POM_HD void pop_flame_ring(uint8_t* r)                               /* PopElem, bboard.hpp:131-137 */
{
    r[R_FINDEX] = uint8_t(ring20(r[R_FINDEX] + 1u));
    r[R_FCOUNT] = uint8_t(r[R_FCOUNT] - 1);
}

/* ---------------------------------------------------------------------------------------------
 * Ray-parallel form of ExplodeTopBomb (bboard.cpp:191-196) -> SpawnFlame (:198-263) for the warp-cooperative
 * tick (pom_kernels.cuh, warp_explode_due): four lanes own the four rays of one explosion.
 * The rays of one spawn touch disjoint cells, so they only interact through a chained explosion
 * (SpawnFlameItem finds a bomb queue entry on the cell, :30-39): the nested spawn writes cells that later
 * rays of the parent - or rays of a grand-child - may cross.  So every ray is first SCANNED without writing
 * (ray_scan); when no ray meets a bomb the four rays are COMMITTED independently (ray_commit) and three lanes
 * share the spawn's prologue, the kills and PopBomb (top_bomb_commit_part); otherwise nothing has been written and
 * the explosion runs on the serial machine (`explode`).  In the bench workload 0.2 % of the explosions chain;
 * in the kick/bomb stress regime most do.
 *
 * Plan word of a ray: bits 0-3 cells that become flame, bits 4-6 = 1 | flag << 1 when the last of them was wood
 * (its powerup flag travels into the flame cell, :46-50), bits 8-11 agents killed, bit 12 chain.
 * ------------------------------------------------------------------------------------------- */
enum { RAY_N_MASK = 0xF, RAY_WOOD_SHIFT = 4, RAY_KILL_SHIFT = 8, RAY_KILL_MASK = 0xF00, RAY_CHAIN = 0x1000 };

POM_HD uint32_t ray_scan(uint8_t* r, uint32_t ci, int stride, uint32_t len)
{
    uint32_t n = 0, plan = 0;
    POM_LOOP
    for(uint32_t k = 0; k < len; k++)
    {
        ci = uint32_t(int(ci) + stride);
        const uint32_t c = r[R_BOARD + ci];
        if(c == uint32_t(C_RIGID)) break;                             /* :53-56 */
        if(c_is_wood(c))                                              /* :45-51 */
        {
            n++;
            plan |= (1u | (((c - 2u) & 3u) << 1)) << RAY_WOOD_SHIFT;
            break;
        }
        const bool isAgent = c_is_agent(c);
        if(isAgent) plan |= (1u << RAY_KILL_SHIFT) << (c - uint32_t(C_AGENT0));
        if((isAgent || c == uint32_t(C_BOMB)) && bomb_index(r, (ci % 11u) | ((ci / 11u) << 4)) >= 0)
        {
            plan |= RAY_CHAIN;                                        /* :30-39 */
            break;
        }
        n++;
    }
    return plan | n;
}

POM_HD void ray_commit(uint8_t* r, uint32_t ci, int stride, uint32_t plan, uint32_t slot)
{
    const uint32_t n = plan & RAY_N_MASK;
    const uint32_t code = uint32_t(C_FLAME) | (slot << 2);
    POM_LOOP
    for(uint32_t k = 0; k < n; k++)
    {
        ci = uint32_t(int(ci) + stride);
        r[R_BOARD + ci] = uint8_t(code);
    }
    if(plan & (1u << RAY_WOOD_SHIFT)) r[R_BOARD + ci] = uint8_t(code | ((plan >> (RAY_WOOD_SHIFT + 1)) & 3u));
}

/* The part of a chain-free ExplodeTopBomb that is not a ray, in three pieces that touch disjoint fields of the record,
 * so that three lanes of the group can run them at once:
 *   part 0  SpawnFlame's prologue (bboard.cpp:200-208): the flame-queue entry
 *   part 1  the origin cell (:210-217) and the kills of the whole spawn (State::Kill, bboard.hpp:474-481;
 *           `ray_kills` = the four ray plans OR-ed)
 *   part 2  PopBomb (:93-97)
 * `c` = the top bomb word and `slot` = the flame-ring slot the spawn takes, both read before any part ran.
 * Returns true when the flame ring was already full (F_FLAME_OVF). */
POM_HD bool top_bomb_commit_part(uint8_t* r, uint32_t c, uint32_t ray_kills, uint32_t part, uint32_t slot)
{
    const uint32_t p = c & 0xFFu;
    bool overflow = false;
    if(part == 0u)
    {
        const uint32_t fc = r[R_FCOUNT];
        overflow = fc >= 20u;
        r[R_FPOS + slot] = uint8_t(p);
        r[R_FSTR + slot] = uint8_t((c >> 12) & 15u);
        r[R_FTIME + slot] = uint8_t(POM_FLAME_LIFETIME);
        r[R_FCOUNT] = uint8_t(fc + 1u);
    }
    else if(part == 1u)
    {
        uint8_t* cell = r + R_BOARD + cell_of(p);
        uint32_t kills = (ray_kills & RAY_KILL_MASK) >> RAY_KILL_SHIFT;
        const uint32_t co = *cell;
        if(c_is_agent(co)) kills |= 1u << (co - uint32_t(C_AGENT0));
        *cell = uint8_t(C_FLAME | (slot << 2));
        if(kills)
        {
            /* bit a of kills -> AF_DEAD in byte a; agents already dead are not counted twice */
            uint32_t* aw = reinterpret_cast<uint32_t*>(r + R_APOS);
            const uint32_t deadBits = ((kills & 1u) << 1) | ((kills & 2u) << 8) | ((kills & 4u) << 15) | ((kills & 8u) << 22);
            const uint32_t fresh = deadBits & ~aw[4];
            aw[4] |= fresh;
            r[R_ALIVE] = uint8_t(r[R_ALIVE] - popcount32(fresh));
        }
    }
    else if(part == 2u)
    {
        const int id = int((c >> 8) & 3u);
        r[R_ABCNT + id] = uint8_t(r[R_ABCNT + id] - 1);
        r[R_BINDEX] = uint8_t(ring_next(r[R_BINDEX]));
        r[R_BCOUNT] = uint8_t(r[R_BCOUNT] - 1);
    }
    return overflow;
}

/* whether TickBombs' explosion loop (step_utility.cpp:231-244) has another turn: bombs[0] has timed out */
POM_HD bool top_bomb_due(const uint8_t* r)
{
    return r[R_BCOUNT] > 0 && ((reinterpret_cast<const uint32_t*>(r + R_BOMBS)[r[R_BINDEX]] >> 16) & 15u) == 0u;
}

/* one turn of that loop in the ray-parallel form, the four rays run one after the other: what the four lanes of
 * warp_explode_due do together.  Returns false, having written nothing, when a ray meets a bomb. */
POM_HD bool explode_top_by_rays(uint8_t* r, int& flags)
{
    const uint32_t c = bomb_slot(r, r[R_BINDEX]);
    const uint32_t p = c & 0xFFu, strength = (c >> 12) & 15u;
    const uint32_t ci0 = uint32_t(cell_of(p));
    const uint32_t slot = ring20(r[R_FINDEX] + r[R_FCOUNT]);
    uint32_t plan[4], all = 0;
    int stride[4];
    for(uint32_t d = 0; d < 4; d++)
    {
        const uint32_t len = ray_length(p, strength, d, stride[d]);
        plan[d] = ray_scan(r, ci0, stride[d], len);
        all |= plan[d];
    }
    if(all & RAY_CHAIN) return false;
    for(uint32_t d = 0; d < 4; d++)
    {
        ray_commit(r, ci0, stride[d], plan[d], slot);
        if(top_bomb_commit_part(r, c, all, d, slot)) flags |= F_FLAME_OVF;
    }
    return true;
}

/* bboard::Step with the explosion loop in the ray-parallel form (host emulation of the warp-cooperative tick) */
POM_HD int step_by_rays(uint8_t* r, uint32_t moves)
{
    if(flames_age(r))
    {
        const int n = r[R_FCOUNT];
        for(int i = 0; i < n && r[R_FTIME + r[R_FINDEX]] == 0; i++)
        {
            for(uint32_t d = 0; d < 4; d++) pop_flame_arm(r, d);
            pop_flame_ring(r);
        }
    }
    bool due;
    int flags = step_body(r, moves, due, false);
    if(due)
    {
        const int bc = r[R_BCOUNT];
        for(int k = 0; k < bc && top_bomb_due(r); k++)
        {
            if(!explode_top_by_rays(r, flags))
            {
                flags |= step_explode_due(r);                          /* serial machine: finishes the loop */
                break;
            }
        }
    }
    return flags;
}

/* bboard::Step, step.cpp:9-284 */
POM_HD int step(uint8_t* r, uint32_t moves)
{
    tick_flames(r);                                                  /* :15 */
    bool due;
    return step_body(r, moves, due, true);
}

/* Environment::Step's bookkeeping after bboard::Step (environment.cpp:150-168).
 * TEAMS: the 2v2 team game (team 0 = agents 0 and 2, team 1 = agents 1 and 3; the reference has no team mode, so this
 * is the project's definition).  A team is alive while one of its agents is; the per-agent dead flags decide, not the
 * aliveAgents counter (the two agree in every state reachable from InitState).  One team left: DONE, and the winner
 * field holds the team index; none left: DONE | DRAW; both: the game goes on. */
template<bool TEAMS = false>
POM_HD void env_post(uint8_t* r)
{
    uint32_t st = r[R_STATUS];
    uint16_t* ts = reinterpret_cast<uint16_t*>(r + R_TIME);
    /* timeStep is 16 bits in the record (an int in the reference): a game that would pass 65535 ticks leaves what the
     * record can carry, exactly like an upload with timeStep > 65535 (pack) */
    if(*ts == 0xFFFFu) st |= POM_STATUS_INVALID;
    else *ts = uint16_t(*ts + 1);
    if(TEAMS)
    {
        const bool a0 = !(r[R_AFLAGS + 0] & AF_DEAD) || !(r[R_AFLAGS + 2] & AF_DEAD);
        const bool a1 = !(r[R_AFLAGS + 1] & AF_DEAD) || !(r[R_AFLAGS + 3] & AF_DEAD);
        if(a0 != a1) st = (st & POM_STATUS_INVALID) | POM_STATUS_DONE | ((a0 ? 0u : 1u) << POM_STATUS_WINNER_SHIFT);
        else if(!a0) st = (st & POM_STATUS_INVALID) | POM_STATUS_DONE | POM_STATUS_DRAW;
        r[R_STATUS] = uint8_t(st);
        return;
    }
    const int alive = int(int8_t(r[R_ALIVE]));
    if(alive == 1)
    {
        uint32_t w = 0;
        for(uint32_t a = 0; a < 4; a++)
        {
            if(!(r[R_AFLAGS + a] & AF_DEAD)) w = a;
        }
        st = (st & POM_STATUS_INVALID) | POM_STATUS_DONE | (w << POM_STATUS_WINNER_SHIFT);
    }
    if(alive == 0) st = (st & POM_STATUS_INVALID) | POM_STATUS_DONE | POM_STATUS_DRAW;
    r[R_STATUS] = uint8_t(st);
}

/* Environment::Step on the record (environment.cpp:125-128,149-168): skip finished envs, Step,
 * timeStep++, winner / draw (TEAMS: the team game's rule, env_post).  Returns F_* flags (0 for a skipped env). */
template<bool TEAMS = false>
POM_HD int env_step(uint8_t* r, uint32_t moves, int invalid_mask = F_INVALID_MASK)
{
    if(r[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID)) return 0;   /* invalid envs freeze: the reference would have crashed */
    const int flags = step(r, moves);
    if(flags & invalid_mask) r[R_STATUS] |= POM_STATUS_INVALID;
    env_post<TEAMS>(r);
    return flags;
}

/* The per-agent reward of one tick (pom_batch_step_rewards; the reference has no reward, so this is the project's
 * definition, after the reward function of the Pommerman Python environment).  Byte a of the result is r[a] as an int8:
 *   not stepped (the env was done or invalid when the tick started)   0 for everyone
 *   st & INVALID                                                       0 for everyone (aborted episode, no outcome)
 *   DONE, winner w                        +1 for w (team game: both agents of team w), -1 for the others
 *   DONE | DRAW, or TRUNCATED                                         -1 for everyone
 *   running        free-for-all: -1 for a dead agent, 0 for a live one; team game: 0 for everyone
 * `st` is the end-of-tick status byte BEFORE any auto-reset (what status_out reports); `aflags` the record's agent-flags
 * word after the tick.  TRUNCATED is only set when DONE is not, so a win on the last allowed tick is a win.  aflags is
 * read only while the game runs, and a running env is never reset: the word may come from the record after the reset. */
template<bool TEAMS = false>
POM_HD uint32_t tick_rewards(bool stepped, uint32_t st, uint32_t aflags)
{
    if(!stepped || (st & POM_STATUS_INVALID)) return 0u;
    if((st & (POM_STATUS_DONE | POM_STATUS_DRAW)) == POM_STATUS_DONE)
    {
        const uint32_t w = (st & POM_STATUS_WINNER_MASK) >> POM_STATUS_WINNER_SHIFT;
        const uint32_t win = TEAMS ? (0x00FF00FFu << (8u * (w & 1u))) : (0xFFu << (8u * w));
        return (0xFFFFFFFFu & ~win) | (0x01010101u & win);
    }
    if(st & (POM_STATUS_DONE | POM_STATUS_TRUNCATED)) return 0xFFFFFFFFu;
    if(TEAMS) return 0u;
    return ((aflags >> 1) & 0x01010101u) * 0xFFu;                    /* AF_DEAD = bit 1 of each agent's byte */
}

/* The team radio (POM_INIT_RADIO; after the team-radio environment of Pommerman, pommerman/envs/v2.py).  Record bytes
 * R_RADIO..R_RADIO + 2, zero padding on every other handle, hold each agent's last message: two words w0, w1 of 0..7 as
 * the 6-bit value w0 | w1 << 3, agent a in bits 6a..6a+5 of the little-endian 24-bit value. */
POM_HD uint32_t radio_message(const uint8_t* r, int agent)
{
    const uint32_t v = uint32_t(r[R_RADIO]) | (uint32_t(r[R_RADIO + 1]) << 8) | (uint32_t(r[R_RADIO + 2]) << 16);
    return (v >> (6 * agent)) & 63u;
}

/* the latch of a tick that steps the env (pom_batch_step_radio): byte a of `msgs` (bits 0..5) becomes agent a's last
 * message if a's dead flag is clear, (0, 0) if it is set.  Run BEFORE the tick, on the start-of-tick dead flags: an agent
 * that dies in this tick still gets its message through (Pommerman checks `not agent.is_alive` before stepping).  An
 * auto-reset after the tick overwrites the bytes with the template's zeros. */
POM_HD void radio_latch(uint8_t* r, uint32_t msgs)
{
    const uint32_t aflags = *reinterpret_cast<const uint32_t*>(r + R_AFLAGS);
    uint32_t v = 0u;
    for(int a = 0; a < 4; a++)
        if(!((aflags >> (8 * a)) & AF_DEAD)) v |= ((msgs >> (8 * a)) & 63u) << (6 * a);
    r[R_RADIO] = uint8_t(v);
    r[R_RADIO + 1] = uint8_t(v >> 8);
    r[R_RADIO + 2] = uint8_t(v >> 16);
}

/* the scalar word of an observation that holds "observer alive" in its byte 0 gets the teammate's (agent ^ 2) last
 * message in bytes 1 and 2: w0, then w1 */
POM_HD uint32_t radio_obs_bytes(const uint8_t* r, int agent)
{
    const uint32_t m = radio_message(r, agent ^ 2);
    return ((m & 7u) << 8) | ((m >> 3) << 16);
}

/* ---------------------------------------------------------------------------------------------
 * AoS <-> record converters (K5).  pack() returns 0, or a non-zero reason when the AoS state holds
 * a value the record cannot carry (the env is then marked POM_STATUS_INVALID).
 * ------------------------------------------------------------------------------------------- */
POM_HD int pack(const pom_state* s, uint8_t status, uint8_t* r)
{
    int bad = 0;
    /* rings first: flame cells need the flame queue */
    r[R_BCOUNT] = uint8_t(s->bombs_count);
    r[R_BINDEX] = uint8_t(s->bombs_index);
    if(uint32_t(s->bombs_count) > 20u || uint32_t(s->bombs_index) >= 20u) bad = 1;
    for(int k = 0; k < 20; k++) bomb_slot(r, k) = uint32_t(s->bombs[k]);
    r[R_FCOUNT] = uint8_t(s->flames_count);
    r[R_FINDEX] = uint8_t(s->flames_index);
    if(uint32_t(s->flames_count) > 20u || uint32_t(s->flames_index) >= 20u) bad = 2;
    for(int k = 0; k < 20; k++)
    {
        const pom_flame& f = s->flames[k];
        if(uint32_t(f.x) > 10u || uint32_t(f.y) > 10u || f.timeLeft < -16 || f.timeLeft > 100 || uint32_t(f.strength) > 255u) bad = 3;
        r[R_FPOS + k] = uint8_t((f.x & 15) | ((f.y & 15) << 4));
        r[R_FTIME + k] = uint8_t(f.timeLeft);
        r[R_FSTR + k] = uint8_t(f.strength);
    }
    for(int a = 0; a < 4; a++)
    {
        const pom_agent& g = s->agents[a];
        /* bombCount moves by one per plant / explosion and the ring holds 20 bombs: +-64 leaves the signed byte ample room */
        if(uint32_t(g.x) > 10u || uint32_t(g.y) > 10u || g.bombCount < -64 || g.bombCount > 64 ||
                uint32_t(g.maxBombCount) > 255u || uint32_t(g.bombStrength) > 255u) bad = 4;
        r[R_APOS + a] = uint8_t((g.x & 15) | ((g.y & 15) << 4));
        r[R_ABCNT + a] = uint8_t(g.bombCount);
        r[R_AMAX + a] = uint8_t(g.maxBombCount);
        r[R_ASTR + a] = uint8_t(g.bombStrength);
        r[R_AFLAGS + a] = uint8_t((g.canKick ? AF_CANKICK : 0) | (g.dead ? AF_DEAD : 0));
    }
    if(uint32_t(s->timeStep) > 65535u) bad = 5;
    *reinterpret_cast<uint16_t*>(r + R_TIME) = uint16_t(s->timeStep);
    if(s->aliveAgents < -128 || s->aliveAgents > 127) bad = 6;
    r[R_ALIVE] = uint8_t(s->aliveAgents);
    const int fcount = s->flames_count, findex = s->flames_index;
    for(int c = 0; c < POM_BOARD_CELLS; c++)
    {
        const int v = (&s->board[0][0])[c];
        uint32_t code = 0;
        if(v >= 0 && v <= 9)
        {
            /* PASSAGE RIGID - BOMB - FOG EXTRABOMB INCRRANGE KICK AGENTDUMMY */
            const uint8_t map[10] = { C_PASSAGE, C_RIGID, 0xFF, C_BOMB, 0xFF, C_FOG, C_EXTRABOMB, C_INCRRANGE, C_KICK, C_AGENTDUMMY };
            code = map[v];
            if(code == 0xFFu) { bad = 7; code = 0; }
        }
        else if(v >= POM_ITEM_WOOD && v <= POM_ITEM_WOOD + 4) code = uint32_t(C_WOOD + (v - POM_ITEM_WOOD));
        else if(v >= POM_ITEM_AGENT0 && v <= POM_ITEM_AGENT0 + 3) code = uint32_t(C_AGENT0 + (v - POM_ITEM_AGENT0));
        else if((v >> 16) == 4 && (v & 4) == 0 && ((v & 0xFFFF) >> 3) < POM_BOARD_CELLS)
        {
            const int id = (v & 0xFFFF) >> 3;
            const uint32_t op = uint32_t(id % 11) | (uint32_t(id / 11) << 4);
            int slot = -1;
            for(int k = 0; k < fcount && k < 20; k++)
            {
                const int sl = (findex + k) % 20;
                if(r[R_FPOS + sl] == op) { slot = sl; break; }
            }
            if(slot < 0)
            {
                if(id == 0) slot = C_FLAME_ORPHAN_SLOT;
                else { bad = 8; slot = C_FLAME_ORPHAN_SLOT; }
            }
            code = uint32_t(C_FLAME) | (uint32_t(slot) << 2) | uint32_t(v & 3);
        }
        else bad = 9;
        r[R_BOARD + c] = uint8_t(code);
    }
    r[R_STATUS] = uint8_t(status | (bad ? POM_STATUS_INVALID : 0));
    r[289] = r[290] = r[291] = 0;
    return bad;
}

POM_HD uint8_t unpack(const uint8_t* r, pom_state* s)
{
    for(int c = 0; c < POM_BOARD_CELLS; c++)
    {
        const uint32_t code = r[R_BOARD + c];
        int v;
        if(code & 0x80u)
        {
            const uint32_t op = flame_origin(r, code);
            v = POM_ITEM_FLAMES + ((int(op & 15u) + 11 * int(op >> 4)) << 3) + int(code & 3u);
        }
        else if(code <= 1u) v = int(code);
        else if(code <= 6u) v = POM_ITEM_WOOD + int(code) - C_WOOD;
        else if(code == uint32_t(C_BOMB)) v = POM_ITEM_BOMB;
        else if(code == uint32_t(C_FOG)) v = POM_ITEM_FOG;
        else if(code <= 11u) v = POM_ITEM_EXTRABOMB + int(code) - C_EXTRABOMB;
        else if(code == uint32_t(C_AGENTDUMMY)) v = POM_ITEM_AGENTDUMMY;
        else v = POM_ITEM_AGENT0 + int(code) - C_AGENT0;
        (&s->board[0][0])[c] = v;
    }
    s->timeStep = *reinterpret_cast<const uint16_t*>(r + R_TIME);
    s->aliveAgents = int(int8_t(r[R_ALIVE]));
    for(int a = 0; a < 4; a++)
    {
        pom_agent& g = s->agents[a];
        g.x = r[R_APOS + a] & 15;
        g.y = r[R_APOS + a] >> 4;
        g.bombCount = int(int8_t(r[R_ABCNT + a]));
        g.maxBombCount = r[R_AMAX + a];
        g.bombStrength = r[R_ASTR + a];
        g.canKick = (r[R_AFLAGS + a] & AF_CANKICK) ? 1 : 0;
        g.dead = (r[R_AFLAGS + a] & AF_DEAD) ? 1 : 0;
        g._pad[0] = g._pad[1] = 0;
    }
    for(int k = 0; k < 20; k++) s->bombs[k] = int32_t(reinterpret_cast<const uint32_t*>(r + R_BOMBS)[k]);
    s->bombs_index = r[R_BINDEX];
    s->bombs_count = r[R_BCOUNT];
    for(int k = 0; k < 20; k++)
    {
        pom_flame& f = s->flames[k];
        f.x = r[R_FPOS + k] & 15;
        f.y = r[R_FPOS + k] >> 4;
        f.timeLeft = int(int8_t(r[R_FTIME + k]));
        f.strength = r[R_FSTR + k];
    }
    s->flames_index = r[R_FINDEX];
    s->flames_count = r[R_FCOUNT];
    return r[R_STATUS];
}

/* ---------------------------------------------------------------------------------------------
 * Partial observability (SURVEY §8f row 4).  The reference reserves Item::FOG (bboard.hpp:62) and says that
 * Agent::act receives a "(potentially fogged) board state" (bboard.hpp:529) in which the AgentInfo of agents out of
 * sight is simply not exposed (bboard.hpp:218-226), but it never implements the fogging.  This is Pommerman's rule
 * (a square window of `view` cells around the observer, 4 in the game) applied to a State:
 *   board     cells outside the window become FOG
 *   agents    the observer's own entry is kept; another agent that is dead or stands outside the window keeps only
 *             its `dead` flag: x = y = -1, the other fields 0 (who is alive is public in Pommerman)
 *   bombs     entries outside the window are dropped, the ring is rewritten from slot 0 in logical order
 *   flames    entries whose origin is outside the window are dropped likewise
 *   timeStep, aliveAgents are public
 * ------------------------------------------------------------------------------------------- */
POM_HD void fog_state(pom_state* s, int agent, int view)
{
    const int ax = s->agents[agent].x, ay = s->agents[agent].y;
    const int x0 = ax - view, x1 = ax + view, y0 = ay - view, y1 = ay + view;
    for(int y = 0; y < POM_BOARD_SIZE; y++)
        for(int x = 0; x < POM_BOARD_SIZE; x++)
            if(x < x0 || x > x1 || y < y0 || y > y1) s->board[y][x] = POM_ITEM_FOG;
    for(int i = 0; i < POM_AGENT_COUNT; i++)
    {
        pom_agent& g = s->agents[i];
        if(i == agent) continue;
        if(g.dead || g.x < x0 || g.x > x1 || g.y < y0 || g.y > y1)
        {
            g.x = -1; g.y = -1; g.bombCount = 0; g.maxBombCount = 0; g.bombStrength = 0; g.canKick = 0;
        }
    }
    int32_t keep[POM_MAX_BOMBS];
    int nb = 0;
    for(int i = 0; i < s->bombs_count && i < POM_MAX_BOMBS; i++)
    {
        const int32_t b = s->bombs[(s->bombs_index + i) % POM_MAX_BOMBS];
        const int bx = b & 15, by = (b >> 4) & 15;
        if(bx >= x0 && bx <= x1 && by >= y0 && by <= y1) keep[nb++] = b;
    }
    for(int i = 0; i < POM_MAX_BOMBS; i++) s->bombs[i] = i < nb ? keep[i] : 0;
    s->bombs_index = 0;
    s->bombs_count = nb;
    pom_flame fk[POM_MAX_BOMBS];
    int nf = 0;
    for(int i = 0; i < s->flames_count && i < POM_MAX_BOMBS; i++)
    {
        const pom_flame f = s->flames[(s->flames_index + i) % POM_MAX_BOMBS];
        if(f.x >= x0 && f.x <= x1 && f.y >= y0 && f.y <= y1) fk[nf++] = f;
    }
    for(int i = 0; i < POM_MAX_BOMBS; i++)
    {
        if(i < nf) s->flames[i] = fk[i];
        else { s->flames[i].x = 0; s->flames[i].y = 0; s->flames[i].timeLeft = 0; s->flames[i].strength = 0; }
    }
    s->flames_index = 0;
    s->flames_count = nf;
}

/* ---------------------------------------------------------------------------------------------
 * Observation planes (SURVEY §8f row 4): what agent `agent` sees through a window of `view` cells, as POM_OBS_BYTES
 * bytes ready for a network input (include/pom_batch.h describes the layout).  Same visibility rule as fog_state; the
 * board plane uses the reference's Item order (bboard.hpp:54-71) with wood / flame powerup flags hidden, as in the game.
 * ------------------------------------------------------------------------------------------- */
/* 32 bytes of an observation at once: one 256-bit store (STG.256, a full sector) on the device */
POM_HD void obs_store32(uint8_t* out, int chunk, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t e, uint32_t f, uint32_t g, uint32_t h)
{
#if defined(__CUDA_ARCH__)
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(out + 32 * chunk), "r"(a), "r"(b), "r"(c), "r"(d), "r"(e), "r"(f), "r"(g), "r"(h) : "memory");
#else
    uint32_t* w = reinterpret_cast<uint32_t*>(out) + 8 * chunk;
    w[0] = a; w[1] = b; w[2] = c; w[3] = d; w[4] = e; w[5] = f; w[6] = g; w[7] = h;
#endif
}

/* per byte: 0xFF where the top bit is set, else 0.  One PRMT on the device: selector nibble 8 + k = "byte k, its sign
 * replicated over the eight bits" (PTX prmt, default mode; __byte_perm masks that bit away, hence the asm) */
POM_HD uint32_t msb_fill(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %1, 0xBA98;" : "=r"(d) : "r"(x));
    return d;
#else
    return ((x >> 7) & 0x01010101u) * 0xFFu;
#endif
}
/* per bit: a where m is set, else b (one LOP3) */
POM_HD uint32_t sel_bits(uint32_t m, uint32_t a, uint32_t b) { return (m & a) | (~m & b); }

/* the window [x0v, x1v] x [y0v, y1v] (every bound replicated into the four bytes of its word; the upper bounds already
 * carry 0x80 per byte) against four cells whose coordinates sit in the bytes of xs / ys: 0xFF per visible cell.  All
 * values are < 0x80, so (a | 0x80) - b keeps the top bit of a byte exactly when a >= b and never borrows from the
 * byte above. */
POM_HD uint32_t window_mask(uint32_t xs, uint32_t ys, uint32_t x0v, uint32_t x1h, uint32_t y0v, uint32_t y1h)
{
    const uint32_t H = 0x80808080u;
    return msb_fill(((xs | H) - x0v) & (x1h - xs) & ((ys | H) - y0v) & (y1h - ys));
}

/* An observation is written by FOUR parts (i = 0..3; on the device the four lanes of a quad, in tests/hostsim one after
 * the other).  `out` is GLOBAL memory, 32-byte aligned (POM_OBS_BYTES = 512), written as 16 chunks of 32 bytes (whole
 * sectors, nothing is read back); part i writes chunks i, i + 4, i + 8 and i + 12, so one store instruction of a quad
 * covers 128 contiguous bytes and a warp's store touches 8 full lines.  (With one lane per env every lane's 32-byte
 * store was a line of its own: 16 x 32 lines per warp and agent, and the L1 data pipe - 67 % busy - bounded the kernel,
 * not HBM: profiles/k_observe_lines_r2.txt.)  Then the few bytes of visible bombs and flames are patched in.
 * Everything the lanes do together is straight-line, byte-parallel code: per board word one load, the window test on
 * the four cells' coordinates, the item ids by range masks, selects - no branch.  Only the patches loop: once per board
 * word that shows a flame (shared out over the four parts), once per bomb. */
struct ObsWindow {
    int x0, x1, y0, y1;                     /* the window, not clamped */
    uint32_t x0v, x1h, y0v, y1h;            /* clamped to the board, replicated per byte; the upper bounds carry 0x80 per byte */
};

POM_HD ObsWindow obs_window(const uint8_t* r, int agent, int view)
{
    const uint32_t H = 0x80808080u;
    const uint32_t ap = r[R_APOS + agent];
    const int ax = int(ap & 15u), ay = int(ap >> 4);
    if(view > 16) view = 16;                                   /* anything past the board is the whole board */
    ObsWindow W;
    W.x0 = ax - view; W.x1 = ax + view; W.y0 = ay - view; W.y1 = ay + view;
    W.x0v = uint32_t(W.x0 < 0 ? 0 : W.x0) * 0x01010101u; W.x1h = uint32_t(W.x1 > 10 ? 10 : W.x1) * 0x01010101u | H;
    W.y0v = uint32_t(W.y0 < 0 ? 0 : W.y0) * 0x01010101u; W.y1h = uint32_t(W.y1 > 10 ? 10 : W.y1) * 0x01010101u | H;
    return W;
}

/* coordinates of the four cells c0 .. c0+3 (c0 = x + 11 y), one per byte; a row ends inside the word when x + j reaches 11 */
POM_HD void obs_cell_coords(int x, int y, uint32_t& xs, uint32_t& ys)
{
    const uint32_t xr = uint32_t(x) * 0x01010101u + 0x03020100u;
    const uint32_t wrap = msb_fill(xr + 0x75757575u);                               /* x >= 11 */
    xs = xr - (wrap & 0x0B0B0B0Bu);
    ys = uint32_t(y) * 0x01010101u + (wrap & 0x01010101u);
}

/* part i, the chunks: board chunk i (cells 32 i .. 32 i + 31; the item ids come from byte-parallel range tests on the
 * cell codes - 0,1 keep; 2..6 wood -> 2; 7 bomb -> 3; 8.. -> code - 3, i.e. fog 5, powerups 6..8, dummy 9, agents
 * 10..13; flame codes have the top bit set -> 4 - then cells outside the window are overwritten with 5, fog), the empty
 * chunks i + 4 and i + 8 of planes 1-3, and chunk i + 12 (part 3: the scalars).  Returns bit w for every board word w
 * of this chunk that shows a visible flame cell. */
/* RADIO: the observation of a radio handle - bytes 493 and 494 carry the teammate's last message (radio_obs_bytes) */
template<bool RADIO = false>
POM_HD uint32_t observe_part_chunks(const uint8_t* r, int agent, const ObsWindow& W, uint8_t* out, int i)
{
    const uint32_t H = 0x80808080u;
    const uint32_t* bw = reinterpret_cast<const uint32_t*>(r + R_BOARD);
    uint32_t litWords = 0u;
    uint32_t word[8];
    int y = (32 * i) / POM_BOARD_SIZE, x = 32 * i - POM_BOARD_SIZE * y;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for(int k = 0; k < 8; k++)
    {
        const int w = 8 * i + k;
        uint32_t xs, ys;
        obs_cell_coords(x, y, xs, ys);
        x += 4;
        if(x >= POM_BOARD_SIZE) { x -= POM_BOARD_SIZE; y++; }
        const uint32_t vis = window_mask(xs, ys, W.x0v, W.x1h, W.y0v, W.y1h);    /* cells 121.. sit in row 11: never visible */
        const uint32_t codes = bw[w < 31 ? w : 30];
        const uint32_t l = codes & 0x7F7F7F7Fu, burn = msb_fill(codes);
        const uint32_t ge2 = msb_fill(l + 0x7E7E7E7Eu), ge7 = msb_fill(l + 0x79797979u), ge8 = msb_fill(l + 0x78787878u);
        const uint32_t minus3 = ((l | H) - 0x03030303u) & 0x7F7F7F7Fu;               /* per byte, no borrow between bytes */
        uint32_t ids = sel_bits(ge2, 0x02020202u, l);
        ids = sel_bits(ge7, 0x03030303u, ids);
        ids = sel_bits(ge8, minus3, ids);
        ids = sel_bits(burn, 0x04040404u, ids);
        ids = sel_bits(vis, ids, 0x05050505u);
        /* bytes 121..127 are the first cells of the bomb-strength plane */
        word[k] = w < 30 ? ids : (w == 30 ? (ids & 0xFFu) : 0u);
        litWords |= ((burn & vis) != 0u && w < 31 ? 1u : 0u) << w;
    }
    obs_store32(out, i, word[0], word[1], word[2], word[3], word[4], word[5], word[6], word[7]);
    obs_store32(out, i + 4, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u);
    obs_store32(out, i + 8, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u);
    uint32_t s1 = 0u, s2 = 0u, s3 = 0u;
    if(i == 3)
    {
        /* chunk 15 = bytes 480..511: the last flame-plane cells, the twelve scalar bytes, the padding */
        const int ammo = int(r[R_AMAX + agent]) - int(int8_t(r[R_ABCNT + agent]));
        const uint32_t deadw = *reinterpret_cast<const uint32_t*>(r + R_AFLAGS) & (uint32_t(AF_DEAD) * 0x01010101u);
        uint32_t alive = 0;
        for(int a = 0; a < 4; a++) alive |= ((deadw >> (8 * a)) & 0xFFu) ? 0u : (1u << a);
        const uint32_t ap = r[R_APOS + agent];
        s1 = (ap & 15u) | ((ap >> 4) << 8) | (uint32_t(ammo < 0 ? 0 : (ammo > 255 ? 255 : ammo)) << 16) | (uint32_t(r[R_ASTR + agent]) << 24);
        s2 = ((r[R_AFLAGS + agent] & AF_CANKICK) ? 1u : 0u) | (alive << 8) | (uint32_t(r[R_TIME]) << 16) | (uint32_t(r[R_TIME + 1]) << 24);
        s3 = (alive >> agent) & 1u;
        if(RADIO) s3 |= radio_obs_bytes(r, agent);
    }
    obs_store32(out, i + 12, 0u, s1, s2, s3, 0u, 0u, 0u, 0u);
    return litWords;
}

/* part i, the patches; `litWords` = the OR of the four parts' observe_part_chunks results.  The caller orders the four
 * parts' chunk stores before any part's patches (__syncwarp on the device): a flame byte may lie in another part's chunk.
 * Bomb bytes are written by the part that owns their chunk, every part walking the whole queue: a later queue entry on
 * the same cell overwrites an earlier one, which one thread's program order guarantees. */
POM_HD void observe_part_patches(const uint8_t* r, const ObsWindow& W, uint8_t* out, int i, uint32_t litWords)
{
    const uint32_t* bw = reinterpret_cast<const uint32_t*>(r + R_BOARD);
    /* visible flame cells: how long they still burn.  Board word w is looked after by part w % 4. */
    uint32_t mine = litWords & (0x11111111u << i);
    if(mine)
    {
        const int fc = r[R_FCOUNT] < 20 ? r[R_FCOUNT] : 20;
        const uint32_t first = r[R_FINDEX];
        POM_LOOP
        while(mine)
        {
#if defined(__CUDA_ARCH__)
            const int w = __ffs(int(mine)) - 1;
#else
            const int w = __builtin_ctz(mine);
#endif
            mine &= mine - 1u;
            const uint32_t codes = bw[w];
            const int c0 = 4 * w, cy = c0 / POM_BOARD_SIZE, cx = c0 - POM_BOARD_SIZE * cy;
            uint32_t xs, ys;
            obs_cell_coords(cx, cy, xs, ys);
            const uint32_t lit = msb_fill(codes) & window_mask(xs, ys, W.x0v, W.x1h, W.y0v, W.y1h);
            for(int j = 0; j < 4; j++)
            {
                if(!((lit >> (8 * j)) & 1u)) continue;
                /* the flame-queue entry the cell belongs to: the first one, in queue order, with the cell's origin
                 * (the rule State::PopFlame matches cells by, bboard.cpp:160-176) */
                const uint32_t origin = flame_origin(r, (codes >> (8 * j)) & 0xFFu);
                uint32_t slot = first;
                POM_LOOP
                for(int k = 0; k < fc; k++, slot = ring_next(slot))
                {
                    if(r[R_FPOS + slot] == origin)
                    {
                        const int t = int(int8_t(r[R_FTIME + slot]));
                        out[363 + c0 + j] = uint8_t(t < 0 ? 0 : t);
                        break;
                    }
                }
            }
        }
    }
    /* visible bombs: blast strength and timer at their cell */
    {
        const int bc = r[R_BCOUNT] < 20 ? r[R_BCOUNT] : 20;
        uint32_t slot = r[R_BINDEX];
        POM_LOOP
        for(int k = 0; k < bc; k++, slot = ring_next(slot))
        {
            const uint32_t b = reinterpret_cast<const uint32_t*>(r + R_BOMBS)[slot];
            const int bx = int(b & 15u), by = int((b >> 4) & 15u);
            if(bx > 10 || by > 10 || bx < W.x0 || bx > W.x1 || by < W.y0 || by > W.y1) continue;
            const int o1 = 121 + bx + 11 * by, o2 = o1 + 121;
            if(((o1 >> 5) & 3) == i) out[o1] = uint8_t((b >> 12) & 15u);
            if(((o2 >> 5) & 3) == i) out[o2] = uint8_t((b >> 16) & 15u);
        }
    }
}

/* the four parts one after the other (tests/hostsim; not used by the kernels) */
template<bool RADIO = false>
POM_HD void observe_planes(const uint8_t* r, int agent, int view, uint8_t* out)
{
    const ObsWindow W = obs_window(r, agent, view);
    uint32_t lit = 0u;
    for(int i = 0; i < 4; i++) lit |= observe_part_chunks<RADIO>(r, agent, W, out, i);
    for(int i = 0; i < 4; i++) observe_part_patches(r, W, out, i, lit);
}

/* ---------------------------------------------------------------------------------------------
 * The CROPPED layout of the same observation (pom_batch_observe_planes_cropped): only the window, four planes of
 * W x W bytes (W = 2 view + 1, view <= 5) centred on the observer - plane cell (row, col) is board cell
 * (x - view + col, y - view + row) - followed by the twelve scalar bytes, padded to a multiple of 32 bytes
 * (view 4: 4 x 81 + 12 = 336 -> 352 bytes instead of 512).  Window cells that lie off the board hold 5 (fog) in the board
 * plane and 0 elsewhere.  Written by the same four parts as the full layout: part i owns the 32-byte chunks i, i + 4, ...
 * ------------------------------------------------------------------------------------------- */
POM_HD uint32_t obs_cropped_bytes(int view) { const uint32_t w = uint32_t(2 * view + 1); return (4u * w * w + 12u + 31u) & ~31u; }

/* the game's item id of a cell code (see observe_part_chunks) */
POM_HD uint32_t obs_item_id(uint32_t code)
{
    return (code & 0x80u) ? 4u : (code >= 8u ? code - 3u : (code == 7u ? 3u : (code >= 2u ? 2u : code)));
}

/* part i, the chunks.  Returns the mask of this part's board-plane bytes (bit b = byte 32 i + b) that show a flame.
 * RADIO: scalar bytes 9 and 10 carry the teammate's last message, as bytes 493 and 494 of the full layout. */
template<bool RADIO = false>
POM_HD uint32_t observe_cropped_part_chunks(const uint8_t* r, int agent, int view, uint8_t* out, int i)
{
    const int W = 2 * view + 1, W2 = W * W;
    const uint32_t nchunks = obs_cropped_bytes(view) >> 5;
    const uint32_t ap = r[R_APOS + agent];
    const int x0 = int(ap & 15u) - view, y0 = int(ap >> 4) - view;
    uint32_t flames = 0u;
    /* the twelve scalar bytes as three words (the layout of the full record's bytes 484..495) */
    uint32_t sc0 = 0u, sc1 = 0u, sc2 = 0u;
    {
        const int ammo = int(r[R_AMAX + agent]) - int(int8_t(r[R_ABCNT + agent]));
        const uint32_t deadw = *reinterpret_cast<const uint32_t*>(r + R_AFLAGS) & (uint32_t(AF_DEAD) * 0x01010101u);
        uint32_t alive = 0;
        for(int a = 0; a < 4; a++) alive |= ((deadw >> (8 * a)) & 0xFFu) ? 0u : (1u << a);
        sc0 = (ap & 15u) | ((ap >> 4) << 8) | (uint32_t(ammo < 0 ? 0 : (ammo > 255 ? 255 : ammo)) << 16) | (uint32_t(r[R_ASTR + agent]) << 24);
        sc1 = ((r[R_AFLAGS + agent] & AF_CANKICK) ? 1u : 0u) | (alive << 8) | (uint32_t(r[R_TIME]) << 16) | (uint32_t(r[R_TIME + 1]) << 24);
        sc2 = (alive >> agent) & 1u;
        if(RADIO) sc2 |= radio_obs_bytes(r, agent);
    }
    POM_LOOP
    for(uint32_t q = uint32_t(i); q < nchunks; q += 4u)
    {
        uint32_t word[8] = { 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u };
        const int o0 = int(32u * q);
        if(o0 < W2)
        {
            /* board plane: walk the window cells of this chunk, row-major, four to an output word.  No branch per cell: a
             * cell off the board reads a clamped address and its code is replaced by 8, the code of FOG, which maps to the
             * id 5; then the byte-parallel mapping of observe_part_chunks turns the four codes into ids, and bytes behind
             * the plane's last cell are cleared. */
            int row = o0 / W, col = o0 - W * row;
#if defined(__CUDACC__)
#pragma unroll
#endif
            for(int k = 0; k < 8; k++)
            {
                uint32_t codes = 0u, inplane = 0u;
#if defined(__CUDACC__)
#pragma unroll
#endif
                for(int j = 0; j < 4; j++)
                {
                    const int x = x0 + col, y = y0 + row;
                    const bool onboard = uint32_t(x) < 11u && uint32_t(y) < 11u;
                    const int cell = onboard ? x + 11 * y : 0;
                    const uint32_t c = onboard ? uint32_t(r[R_BOARD + cell]) : 8u;
                    codes |= c << (8 * j);
                    inplane |= (o0 + 4 * k + j < W2 ? 0xFFu : 0u) << (8 * j);
                    if(++col == W) { col = 0; row++; }
                }
                const uint32_t H = 0x80808080u;
                const uint32_t l = codes & 0x7F7F7F7Fu, burn = msb_fill(codes);
                const uint32_t ge2 = msb_fill(l + 0x7E7E7E7Eu), ge7 = msb_fill(l + 0x79797979u), ge8 = msb_fill(l + 0x78787878u);
                const uint32_t minus3 = ((l | H) - 0x03030303u) & 0x7F7F7F7Fu;
                uint32_t ids = sel_bits(ge2, 0x02020202u, l);
                ids = sel_bits(ge7, 0x03030303u, ids);
                ids = sel_bits(ge8, minus3, ids);
                ids = sel_bits(burn, 0x04040404u, ids);
                word[k] = ids & inplane;
                /* one bit per flame byte of this word: bits 7, 15, 23, 31 -> bits 0..3 */
                const uint32_t fb = burn & inplane & H;
                flames |= ((((fb >> 7) * 0x01020408u) >> 24) & 0x0Fu) << (4 * k);
            }
        }
        /* the scalars: bytes 4 W2 .. 4 W2 + 11, anywhere in (at most two) chunks */
        {
            const int s0 = 4 * W2 - o0;                                /* position of scalar byte 0 within this chunk (W2 is odd: s0 % 4 == 0) */
#if defined(__CUDACC__)
#pragma unroll
#endif
            for(int k = 0; k < 8; k++)
            {
                const int t = 4 * k - s0;                               /* scalar byte held by byte 0 of word k */
                if(t == 0) word[k] |= sc0; else if(t == 4) word[k] |= sc1; else if(t == 8) word[k] |= sc2;
            }
        }
        obs_store32(out, int(q), word[0], word[1], word[2], word[3], word[4], word[5], word[6], word[7]);
    }
    return flames;
}

/* part i, the patches: the lives of this part's flame cells (their bytes may lie in another part's chunk: the caller
 * orders all chunk stores before any patch), and the bomb bytes that fall into this part's chunks */
POM_HD void observe_cropped_part_patches(const uint8_t* r, int agent, int view, uint8_t* out, int i, uint32_t flames)
{
    const int W = 2 * view + 1, W2 = W * W;
    const uint32_t ap = r[R_APOS + agent];
    const int x0 = int(ap & 15u) - view, y0 = int(ap >> 4) - view;
    if(flames)
    {
        const int fc = r[R_FCOUNT] < 20 ? r[R_FCOUNT] : 20;
        const uint32_t first = r[R_FINDEX];
        POM_LOOP
        while(flames)
        {
#if defined(__CUDA_ARCH__)
            const int b = __ffs(int(flames)) - 1;
#else
            const int b = __builtin_ctz(flames);
#endif
            flames &= flames - 1u;
            const int o = 32 * i + b, row = o / W, col = o - W * row;
            const uint32_t origin = flame_origin(r, r[R_BOARD + (x0 + col) + 11 * (y0 + row)]);
            uint32_t slot = first;
            POM_LOOP
            for(int k = 0; k < fc; k++, slot = ring_next(slot))
            {
                if(r[R_FPOS + slot] == origin)
                {
                    const int t = int(int8_t(r[R_FTIME + slot]));
                    out[3 * W2 + o] = uint8_t(t < 0 ? 0 : t);
                    break;
                }
            }
        }
    }
    {
        const int bc = r[R_BCOUNT] < 20 ? r[R_BCOUNT] : 20;
        uint32_t slot = r[R_BINDEX];
        POM_LOOP
        for(int k = 0; k < bc; k++, slot = ring_next(slot))
        {
            const uint32_t b = reinterpret_cast<const uint32_t*>(r + R_BOMBS)[slot];
            const int bx = int(b & 15u), by = int((b >> 4) & 15u);
            const int col = bx - x0, row = by - y0;
            if(bx > 10 || by > 10 || uint32_t(col) >= uint32_t(W) || uint32_t(row) >= uint32_t(W)) continue;
            const int o1 = W2 + row * W + col, o2 = o1 + W2;
            if(((o1 >> 5) & 3) == i) out[o1] = uint8_t((b >> 12) & 15u);
            if(((o2 >> 5) & 3) == i) out[o2] = uint8_t((b >> 16) & 15u);
        }
    }
}

/* the four parts one after the other (tests/hostsim; not used by the kernels) */
template<bool RADIO = false>
POM_HD void observe_cropped(const uint8_t* r, int agent, int view, uint8_t* out)
{
    uint32_t fl[4];
    for(int i = 0; i < 4; i++) fl[i] = observe_cropped_part_chunks<RADIO>(r, agent, view, out, i);
    for(int i = 0; i < 4; i++) observe_cropped_part_patches(r, agent, view, out, i, fl[i]);
}

/* the shared stateless action source (same arithmetic as oracle/pom_oracle.c pom_oracle_rng_moves) */
POM_HD uint64_t splitmix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

POM_HD uint32_t rng_moves(uint64_t seed, uint64_t env, uint32_t tick, uint32_t n_actions)
{
    const uint64_t h = splitmix64(splitmix64(seed ^ (env * 0xD6E8FEB86659FD93ull)) + uint64_t(tick));
    uint32_t out = 0;
    for(int a = 0; a < 4; a++)
    {
        const uint32_t lane = uint32_t(h >> (16 * a)) & 0xFFFFu;
        out |= ((lane * n_actions) >> 16) << (8 * a);
    }
    return out;
}

/* ---------------------------------------------------------------------------------------------
 * Board generation (K3): InitBoardItems (bboard.cpp:346-382) + PutAgentsInCorners (:322-333) on a
 * zero-initialised State, written straight into a packed record.  std::mt19937_64 is the standard
 * MT19937-64; uniform_int_distribution<int> is libstdc++ 13's Lemire multiply-high with rejection
 * (bits/uniform_int_dist.h:252-281), which is what the reference binary uses.
 * Returns 1 when the seed draws the inclusive upper bound q.count (reference defect D2: it then
 * reads an uninitialised stack slot) — such seeds are skipped by the template builder.
 * ------------------------------------------------------------------------------------------- */
struct Mt64 { uint64_t mt[312]; int idx; };

POM_HD void mt64_seed(Mt64& g, uint64_t seed)
{
    g.mt[0] = seed;
    for(int i = 1; i < 312; i++) g.mt[i] = 6364136223846793005ull * (g.mt[i - 1] ^ (g.mt[i - 1] >> 62)) + uint64_t(i);
    g.idx = 312;
}

POM_HD uint64_t mt64_next(Mt64& g)
{
    if(g.idx >= 312)
    {
        for(int i = 0; i < 312; i++)
        {
            const uint64_t x = (g.mt[i] & 0xFFFFFFFF80000000ull) | (g.mt[i == 311 ? 0 : i + 1] & 0x7FFFFFFFull);
            const uint64_t xa = (x >> 1) ^ ((x & 1ull) ? 0xB5026F5AA96619E9ull : 0ull);
            g.mt[i] = g.mt[i < 156 ? i + 156 : i - 156] ^ xa;
        }
        g.idx = 0;
    }
    uint64_t y = g.mt[g.idx++];
    y ^= (y >> 29) & 0x5555555555555555ull;
    y ^= (y << 17) & 0x71D67FFFEDA60000ull;
    y ^= (y << 37) & 0xFFF7EEE000000000ull;
    y ^= (y >> 43);
    return y;
}

POM_HD void mul64wide(uint64_t a, uint64_t b, uint64_t& hi, uint64_t& lo)
{
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umul64hi(a, b);
#else
    const unsigned __int128 p = (unsigned __int128)a * b;
    lo = uint64_t(p);
    hi = uint64_t(p >> 64);
#endif
}

POM_HD int uniform_int(Mt64& g, int a, int b)
{
    const uint64_t range = uint64_t(b) - uint64_t(a) + 1ull;
    uint64_t hi, lo;
    mul64wide(mt64_next(g), range, hi, lo);
    if(lo < range)
    {
        const uint64_t threshold = (0ull - range) % range;
        while(lo < threshold) mul64wide(mt64_next(g), range, hi, lo);
    }
    return a + int(hi);
}

/* zero-initialised State + InitBoardItems(seed); returns the D2 flag */
POM_HD int init_board(uint8_t* r, Mt64& g, int seed)
{
    for(int k = 0; k < POM_REC_BYTES; k++) r[k] = 0;
    for(int k = 0; k < 20; k++) r[R_FTIME + k] = uint8_t(POM_FLAME_LIFETIME);   /* Flame::timeLeft default, bboard.hpp:345 */
    for(int a = 0; a < 4; a++) { r[R_AMAX + a] = 1; r[R_ASTR + a] = POM_BOMB_DEFAULT_STRENGTH; }
    r[R_ALIVE] = 4;

    mt64_seed(g, uint64_t(int64_t(seed)));
    uint8_t q[POM_BOARD_CELLS];
    int count = 0;
    for(int c = 0; c < POM_BOARD_CELLS; c++)
    {
        const int tmp = uniform_int(g, 0, 6);                        /* ChooseItemOuter, bboard.cpp:59-74 */
        const uint8_t item = tmp == 2 ? uint8_t(C_WOOD) : (tmp == 1 ? uint8_t(C_RIGID) : uint8_t(C_PASSAGE));
        r[R_BOARD + c] = item;
        if(item == C_WOOD) q[count++] = uint8_t(c);
    }
    int dirty = 0, total = 0;
    for(;;)
    {
        const int k = uniform_int(g, 0, count);                      /* inclusive bound: D2 when k == count */
        if(k == count) { dirty = 1; break; }
        const int idx = q[k];
        if(r[R_BOARD + idx] == C_WOOD)                               /* (board & 0xFF) == 0: wood without flag */
        {
            r[R_BOARD + idx] = uint8_t(C_WOOD + uniform_int(g, 1, 4));
            total++;
        }
        if(float(total) >= float(count) / 2) break;
    }
    return dirty;
}

/* State::PutAgentsInCorners, bboard.cpp:322-333 (relies on zeroed agent coordinates, as the reference does) */
POM_HD void put_agents_in_corners(uint8_t* r, int a0, int a1, int a2, int a3)
{
    r[R_BOARD + 0] = uint8_t(C_AGENT0 + a0);
    r[R_BOARD + 10] = uint8_t(C_AGENT0 + a1);
    r[R_BOARD + 120] = uint8_t(C_AGENT0 + a2);
    r[R_BOARD + 110] = uint8_t(C_AGENT0 + a3);
    r[R_APOS + a1] = uint8_t((r[R_APOS + a1] & 0xF0) | 10);
    r[R_APOS + a2] = uint8_t(10 | (10 << 4));
    r[R_APOS + a3] = uint8_t((r[R_APOS + a3] & 0x0F) | (10 << 4));
}

/* InitState (bboard.cpp:339-344) on a zero-initialised State */
POM_HD int init_record(uint8_t* r, Mt64& g, int seed, int a0, int a1, int a2, int a3)
{
    const int dirty = init_board(r, g, seed);
    put_agents_in_corners(r, a0, a1, a2, a3);
    return dirty;
}

}

#endif
