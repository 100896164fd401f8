/*
 * fogsim.cpp — TEST-ONLY host build of the FOG instantiation of the device SimpleAgent (pompolicy::simple_moves and
 * simple_act with FOG = true, free-for-all and team-aware), for tests/test_policy_fog.py.  Records are packed and
 * unpacked with tests/hostsim; this file only adds the fogged entry points.  Not part of the product.
 */
#include <cstdint>
#include <cstring>
#include "pom_core.cuh"
#include "pom_policy.cuh"

extern "C" {

/* the device SimpleAgent under fog of war (view >= 0) on packed records, as hostsim_simple_moves */
void fogsim_simple_moves(const uint8_t* recs, long n, pom_simple_agent* A, uint64_t seed, uint64_t env0, uint32_t tick,
                         uint32_t mask, int view, int teams, uint8_t* moves)
{
    for(long e = 0; e < n; e++)
    {
        const uint8_t* r = recs + e * POM_REC_BYTES;
        if(r[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID)) continue;
        uint32_t m;
        std::memcpy(&m, moves + 4 * e, 4);
        pompolicy::SimpleSt st[4];
        std::memcpy(st, A + 4 * e, sizeof st);
        pompolicy::ArrayStore store{ st };
        const uint32_t draws = pomcore::rng_moves(seed, env0 + uint64_t(e), tick, 5);
        m = teams ? pompolicy::simple_moves<true, true>(r, mask, m, draws, store, view)
                  : pompolicy::simple_moves<false, true>(r, mask, m, draws, store, view);
        std::memcpy(A + 4 * e, st, sizeof st);
        std::memcpy(moves + 4 * e, &m, 4);
    }
}

/* SimpleAgent::act for one agent of one packed record under fog of war (k_policy_act's body) */
int fogsim_simple_act(const uint8_t* rec, int agent, pom_simple_agent* mem, int draw, int view, int teams)
{
    const pompolicy::Boards B = pompolicy::make_boards(rec);
    pompolicy::SimpleSt st;
    std::memcpy(&st, mem, sizeof st);
    const uint32_t m = teams ? pompolicy::simple_act<true, true>(rec, B, agent, st, uint32_t(draw), view)
                             : pompolicy::simple_act<false, true>(rec, B, agent, st, uint32_t(draw), view);
    std::memcpy(mem, &st, sizeof st);
    return int(m);
}

}
