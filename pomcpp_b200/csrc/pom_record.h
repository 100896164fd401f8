/*
 * pom_record.h — the packed per-env record kept in HBM (and staged in shared memory).
 *
 * One env = 292 bytes = 73 32-bit words.  73 is odd, so when the 32 lanes of a warp touch the
 * same field of 32 consecutive records in shared memory they hit 32 different banks.
 * 289 bytes are payload (SURVEY Appendix B, the figure behind the 582 B/env-step roofline
 * accounting); 3 bytes pad the record to a word multiple.  A radio handle keeps its team messages in
 * those 3 bytes, so the radio adds no byte to what a kernel moves per env.
 *
 * Replaces the reference's 1004-byte AoS `bboard::State` (include/bboard.hpp:356-383).
 *
 *  offset  bytes  field
 *  0       121    board, 1 byte per cell, index = x + 11*y            (State::board, int[11][11])
 *  121     1      bombs.count                                          (FixedQueue::count)
 *  122     1      bombs.index                                          (FixedQueue::index)
 *  123     1      flames.count
 *  124     80     bombs.queue[20], the reference's raw 32-bit Bomb words, PHYSICAL ring order,
 *                 stale slots included (SURVEY Q4)                     (bboard.hpp:261-335)
 *  204     4      agent position, byte a = x | y<<4                    (AgentInfo::x,y)
 *  208     4      agent bombCount, signed byte (goes to -1, SURVEY Q12)
 *  212     4      agent maxBombCount
 *  216     4      agent bombStrength
 *  220     4      agent flags: bit0 canKick, bit1 dead
 *  224     2      timeStep (u16; an env about to pass 65535 is marked POM_STATUS_INVALID instead of wrapping)
 *  226     1      aliveAgents (signed byte)
 *  227     1      status (POM_STATUS_* of include/pom_state.h; the reference keeps these in Environment)
 *  228     20     flames.queue[20].position, x | y<<4, PHYSICAL ring order
 *  248     20     flames.queue[20].timeLeft (signed byte)
 *  268     20     flames.queue[20].strength
 *  288     1      flames.index
 *  289     3      radio (handles made with POM_INIT_RADIO), zero otherwise: the last message of agent a, w0 | w1 << 3
 *                 (two 3-bit words), in bits 6a..6a+5 of the little-endian 24-bit value (pomcore::radio_latch)
 *
 * Cell codes (1 byte, bijective on every value the reference can produce, bboard.hpp:54-71):
 *   0 PASSAGE  1 RIGID  2..6 WOOD+flag(0..4)  7 BOMB  8 FOG  9 EXTRABOMB  10 INCRRANGE  11 KICK
 *   12 AGENTDUMMY  13..16 AGENT0..3
 *   0x80 | slot<<2 | flag : FLAMES whose origin id (x+11y) is flames.queue[slot].position; slot is
 *       the PHYSICAL ring slot 0..19 (stable for the flame's life: flames are only PopElem'd,
 *       bboard.cpp:179); slot 31 = a flame cell with origin id 0 and no queue entry (the literal
 *       Item::FLAMES of unit test board_logic.cpp:504).  PopFlame compares origin POSITIONS, so two
 *       live flames sharing an origin behave as in the reference (bboard.cpp:160-176).
 */
#ifndef POM_RECORD_H_
#define POM_RECORD_H_

#include <stdint.h>

#define POM_REC_BYTES   292
#define POM_REC_WORDS   73
#define POM_REC_PAYLOAD 289

enum {
    R_BOARD  = 0,
    R_BCOUNT = 121,
    R_BINDEX = 122,
    R_FCOUNT = 123,
    R_BOMBS  = 124,
    R_APOS   = 204,
    R_ABCNT  = 208,
    R_AMAX   = 212,
    R_ASTR   = 216,
    R_AFLAGS = 220,
    R_TIME   = 224,
    R_ALIVE  = 226,
    R_STATUS = 227,
    R_FPOS   = 228,
    R_FTIME  = 248,
    R_FSTR   = 268,
    R_FINDEX = 288,
    R_RADIO  = 289
};

enum {
    C_PASSAGE = 0, C_RIGID = 1, C_WOOD = 2, C_BOMB = 7, C_FOG = 8,
    C_EXTRABOMB = 9, C_INCRRANGE = 10, C_KICK = 11, C_AGENTDUMMY = 12, C_AGENT0 = 13,
    C_FLAME = 0x80, C_FLAME_ORPHAN_SLOT = 31
};

enum { AF_CANKICK = 1, AF_DEAD = 2 };

#endif
