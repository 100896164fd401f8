/*
 * teamsim.cpp — TEST-ONLY host build of the 2v2 team game's instantiation of the device code (pomcore::env_step<true>,
 * pomcore::env_post<true>, pompolicy::simple_moves<true>), for tests/test_teams.py.  Records are packed and unpacked
 * with tests/hostsim; this file only adds the TEAMS entry points.  Not part of the product.
 */
#include <cstdint>
#include <cstring>
#include "pom_core.cuh"
#include "pom_policy.cuh"

extern "C" {

/* Environment::Step with the team game's episode rule on packed records.  by_rays != 0: the tick in the decomposition
 * of the warp-cooperative kernels (pomcore::step_by_rays) */
void teamsim_step_records(uint8_t* recs, long n, const uint8_t* moves, int by_rays, uint8_t* flags_out)
{
    for(long e = 0; e < n; e++)
    {
        uint32_t m;
        std::memcpy(&m, moves + 4 * e, 4);
        uint8_t* r = recs + e * POM_REC_BYTES;
        int f = 0;
        if(!by_rays) f = pomcore::env_step<true>(r, m);
        else if(!(r[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID)))
        {
            f = pomcore::step_by_rays(r, m);
            if(f & pomcore::F_INVALID_MASK) r[R_STATUS] |= POM_STATUS_INVALID;
            pomcore::env_post<true>(r);
        }
        if(flags_out) flags_out[e] = uint8_t(f);
    }
}

/* the team-aware device SimpleAgent on packed records (as hostsim_simple_moves for free-for-all) */
void teamsim_simple_moves(const uint8_t* recs, long n, pom_simple_agent* A, uint64_t seed, uint64_t env0, uint32_t tick,
                          uint32_t mask, uint8_t* moves)
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
        m = pompolicy::simple_moves<true>(r, mask, m, pomcore::rng_moves(seed, env0 + uint64_t(e), tick, 5), store);
        std::memcpy(A + 4 * e, st, sizeof st);
        std::memcpy(moves + 4 * e, &m, 4);
    }
}

}
