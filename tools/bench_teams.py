"""Throughput of the 2v2 team game (POM_INIT_TEAMS) against free-for-all on one GPU; prints one JSON line per leg and mode.

    python tools/bench_teams.py [--rounds R] [--steps K]

 step      the plain per-tick loop of bench.py: 1 Mi envs, four uniform random agents, pom_batch_step with
           AUTORESET | COUNT, one launch per tick, moves pre-generated on the device (a ring of 256 ticks)
           modes: ffa (the specialised k_step_ws image), ffa_generic (POM_WS_NOSPEC=1: the generic image, which the
           team game runs too), teams
 rollout   bench.py's legs.rollout: the fused 800-tick rollout, 512 Ki envs, in-kernel RNG, auto-reset
           modes: ffa (specialised image), ffa_generic, teams
 simple4   four SimpleAgents per env through pom_batch_rollout (1 Mi envs: k_policy_moves + the per-tick step, tick by
           tick), 200 ticks, auto-reset, 800-tick limit.  modes: ffa, teams

Every working set is larger than the 126 MB L2 (1 Mi records = 306 MB, 512 Ki = 153 MB), so no flush is needed between
timed passes (the convention of bench.py).  The modes of a leg are timed in turn, round after round, so that other load on
the machine falls on all of them alike; each line carries every round's figure and their median.  The episode counters
show why the modes differ besides the kernel: team games end sooner, so there are more auto-resets.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pomcpp_b200 as pb  # noqa: E402

SEED = 20240229
N_STEP, N_ROLL = 1 << 20, 1 << 19
RING = 256


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


def make(n, mode):
    """a handle of the mode: ffa / ffa_generic (POM_WS_NOSPEC=1, read when the handle is made) / teams"""
    if mode == "ffa_generic":
        os.environ["POM_WS_NOSPEC"] = "1"
    try:
        return pb.Batch(n, n_templates=4096, max_ticks=800, teams=mode == "teams")
    finally:
        os.environ.pop("POM_WS_NOSPEC", None)


def counters(b):
    s = b.stats()
    return {"episodes": s.episodes, "mean_episode_len": s.sum_episode_len / max(1, s.episodes), "wins": list(s.wins),
            "draws": s.draws, "truncated": s.truncated, "invalid": s.invalid}


def step_leg(mode, steps):
    b = make(N_STEP, mode)
    moves = b.alloc(4 * N_STEP * RING)
    for t in range(RING):
        b.generate_moves(moves.value + 4 * N_STEP * t, SEED, 100000 + t, 6)
    b.rollout(96, SEED, 0, 0)                          # untimed: the steady-state mix of game phases
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT
    for w in range(20):
        b.step(moves.value + 4 * N_STEP * (w % RING), flags)
    b.sync()
    b.clear_stats()
    b.event(0)
    for k in range(steps):
        b.step(moves.value + 4 * N_STEP * ((20 + k) % RING), flags)
    b.event(1)
    ms = b.elapsed_ms() / steps
    c = counters(b)
    assert b.stats().env_steps == N_STEP * steps
    b.free(moves)
    b.close()
    return {"ms_per_tick": ms, "env_steps_per_s": N_STEP / (ms * 1e-3), **c}


def rollout_leg(mode, _):
    b = make(N_ROLL, mode)
    b.rollout(64, SEED, 0, 0)
    b.sync()
    b.clear_stats()
    b.event(0)
    b.rollout(800, SEED, 64, 0)
    b.event(1)
    ms = b.elapsed_ms()
    c = counters(b)
    assert b.stats().env_steps == N_ROLL * 800
    b.close()
    return {"ms": ms, "env_steps_per_s": N_ROLL * 800 / (ms * 1e-3), **c}


def simple4_leg(mode, _):
    b = make(N_STEP, mode)
    b.rollout(40, SEED, 0, pb.ROLL_SIMPLE(15))         # untimed: the games develop, the policy memories exist
    b.sync()
    b.clear_stats()
    b.event(0)
    b.rollout(200, SEED, 40, pb.ROLL_SIMPLE(15))
    b.event(1)
    ms = b.elapsed_ms()
    c = counters(b)
    b.close()
    return {"ms": ms, "env_steps_per_s": N_STEP * 200 / (ms * 1e-3), **c}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    a = ap.parse_args()
    gpu = gpu_info()
    legs = (("step", step_leg, ("ffa", "ffa_generic", "teams")),
            ("rollout", rollout_leg, ("ffa", "ffa_generic", "teams")),
            ("simple4", simple4_leg, ("ffa", "teams")))
    for leg, fn, modes in legs:
        runs = {m: [] for m in modes}
        for _ in range(a.rounds):
            for m in modes:
                runs[m].append(fn(m, a.steps))
        for m in modes:
            rates = sorted(r["env_steps_per_s"] for r in runs[m])
            print(json.dumps({"leg": leg, "mode": m, "env_steps_per_s": rates[len(rates) // 2], "rounds": runs[m],
                              "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
