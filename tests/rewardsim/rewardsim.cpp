/*
 * rewardsim.cpp — TEST-ONLY host build of one tick of pom_batch_step_rewards for tests/test_rewards.py: the tick of the
 * device code (pomcore::env_step<TEAMS>), the per-tick kernel's end of tick (truncation at max_ticks, auto-reset from the
 * template pool, the status byte before the reset) and pomcore::tick_rewards<TEAMS> on the record after it, as k_step_ws
 * runs them.  Records are packed and unpacked with tests/hostsim.  Not part of the product.
 */
#include <cstdint>
#include <cstring>
#include "pom_core.cuh"

template<bool TEAMS>
static void tick(uint8_t* recs, long n, const uint8_t* moves, int autoreset, uint32_t max_ticks,
                 const uint8_t* templates, long n_templates, uint64_t env0, uint32_t* episodes, uint8_t* status_out,
                 uint32_t* rewards)
{
    for(long e = 0; e < n; e++)
    {
        uint8_t* r = recs + e * POM_REC_BYTES;
        uint32_t m;
        std::memcpy(&m, moves + 4 * e, 4);
        const bool stepped = !(r[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID));
        pomcore::env_step<TEAMS>(r, m);
        uint32_t st = r[R_STATUS];
        if(autoreset && stepped)
        {
            /* finish_and_reset (pom_kernels.cuh) */
            uint16_t len;
            std::memcpy(&len, r + R_TIME, 2);
            if(!(st & POM_STATUS_DONE) && max_ticks && len >= max_ticks) st |= POM_STATUS_TRUNCATED;
            if(st & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID))
            {
                const uint32_t ep = ++episodes[e];
                std::memcpy(r, templates + ((env0 + uint64_t(e) + ep) % uint64_t(n_templates)) * POM_REC_BYTES, POM_REC_BYTES);
            }
        }
        status_out[e] = uint8_t(st);
        uint32_t aflags;
        std::memcpy(&aflags, r + R_AFLAGS, 4);
        rewards[e] = pomcore::tick_rewards<TEAMS>(stepped, st, aflags);
    }
}

extern "C" {

void rewardsim_tick(uint8_t* recs, long n, const uint8_t* moves, int teams, int autoreset, uint32_t max_ticks,
                    const uint8_t* templates, long n_templates, uint64_t env0, uint32_t* episodes, uint8_t* status_out,
                    uint32_t* rewards)
{
    if(teams) tick<true>(recs, n, moves, autoreset, max_ticks, templates, n_templates, env0, episodes, status_out, rewards);
    else tick<false>(recs, n, moves, autoreset, max_ticks, templates, n_templates, env0, episodes, status_out, rewards);
}

}
