/*
 * radiosim.cpp — TEST-ONLY host build of one tick of pom_batch_step_radio for tests/test_radio.py: the radio latch
 * (pomcore::radio_latch, before the tick), the team game's tick of the device code (pomcore::env_step<true>), the per-tick
 * kernel's end of tick (truncation at max_ticks, auto-reset from the template pool, the status byte before the reset)
 * and pomcore::tick_rewards<true>, as k_step_ws runs them; and the RADIO observation planes (pomcore::observe_planes<true>,
 * pomcore::observe_cropped<true>).  Records are packed and unpacked with tests/hostsim.  Not part of the product.
 */
#include <cstdint>
#include <cstring>
#include "pom_core.cuh"

extern "C" {

void radiosim_tick(uint8_t* recs, long n, const uint8_t* moves, const uint8_t* msgs, int autoreset, uint32_t max_ticks,
                   const uint8_t* templates, long n_templates, uint64_t env0, uint32_t* episodes, uint8_t* status_out,
                   uint32_t* rewards)
{
    for(long e = 0; e < n; e++)
    {
        uint8_t* r = recs + e * POM_REC_BYTES;
        uint32_t m, msg;
        std::memcpy(&m, moves + 4 * e, 4);
        std::memcpy(&msg, msgs + 4 * e, 4);
        const bool stepped = !(r[R_STATUS] & (POM_STATUS_DONE | POM_STATUS_INVALID));
        if(stepped) pomcore::radio_latch(r, msg);
        pomcore::env_step<true>(r, m);
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
        rewards[e] = pomcore::tick_rewards<true>(stepped, st, aflags);
    }
}

/* the last messages of every record in the pom_batch_radio_download encoding (byte a = agent a's w0 | w1 << 3) */
void radiosim_messages(const uint8_t* recs, long n, uint8_t* out)
{
    for(long e = 0; e < n; e++)
        for(int a = 0; a < 4; a++) out[4 * e + a] = uint8_t(pomcore::radio_message(recs + e * POM_REC_BYTES, a));
}

/* the observation planes of a radio handle, full (cropped = 0) or cropped layout */
void radiosim_observe(const uint8_t* recs, long n, int agent, int view, int cropped, uint8_t* out)
{
    const long rb = cropped ? long(pomcore::obs_cropped_bytes(view)) : 512;
    for(long e = 0; e < n; e++)
    {
        if(cropped) pomcore::observe_cropped<true>(recs + e * POM_REC_BYTES, agent, view, out + rb * e);
        else pomcore::observe_planes<true>(recs + e * POM_REC_BYTES, agent, view, out + rb * e);
    }
}

/* InitState on a zero-initialised record (pomcore::init_record, the device templates' generator): its radio bytes */
void radiosim_init_record_radio(int seed, uint8_t* out3)
{
    uint8_t r[POM_REC_BYTES];
    std::memset(r, 0xA5, sizeof r);
    pomcore::Mt64 g;
    pomcore::init_record(r, g, seed, 0, 1, 2, 3);
    std::memcpy(out3, r + R_RADIO, 3);
}

}
