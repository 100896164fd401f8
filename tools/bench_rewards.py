"""Cost of the per-agent rewards of pom_batch_step_rewards against the plain per-tick step on one GPU; prints one JSON line
per game mode and step mode.

    python tools/bench_rewards.py [--rounds R] [--steps K]

The loop of bench.py: 1 Mi envs, four uniform random agents, AUTORESET | COUNT, one launch per tick, moves from a ring of
256 move sets pre-generated on the device, the rewards (and status bytes) to device buffers.
  game     ffa, teams
  step     step          pom_batch_step (free-for-all: the specialised k_step_ws image)
           step_generic  pom_batch_step on a handle made with POM_WS_NOSPEC=1: the generic image, which the REWARDS
                         image extends (free-for-all only; the team game has no specialised image)
           rewards       pom_batch_step_rewards without status bytes
           rewards_status  pom_batch_step_rewards with status bytes
The record array (1 Mi x 292 B = 306 MB) is larger than the 126 MB L2, so no flush is needed between timed passes.  The
step modes of a game are timed in turn, round after round, so that other load on the machine falls on all of them alike;
each line carries every round's figure and their median, and the card's name, power limit and SM clock read in the run.
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
N = 1 << 20
RING = 256


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


def run(game, mode, steps):
    if mode == "step_generic":
        os.environ["POM_WS_NOSPEC"] = "1"
    try:
        b = pb.Batch(N, n_templates=4096, max_ticks=800, teams=game == "teams")
    finally:
        os.environ.pop("POM_WS_NOSPEC", None)
    moves = b.alloc(4 * N * RING)
    rewards, status = b.alloc(4 * N), b.alloc(N)
    for t in range(RING):
        b.generate_moves(moves.value + 4 * N * t, SEED, 100000 + t, 6)
    b.rollout(96, SEED, 0, 0)                              # untimed: the steady-state mix of game phases
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT

    def tick(k):
        mv = moves.value + 4 * N * (k % RING)
        if mode.startswith("rewards"):
            b.step_rewards(mv, rewards, status if mode == "rewards_status" else None, flags)
        else:
            b.step(mv, flags)
    for w in range(20):
        tick(w)
    b.sync()
    b.clear_stats()
    b.event(0)
    for k in range(steps):
        tick(20 + k)
    b.event(1)
    ms = b.elapsed_ms() / steps
    assert b.stats().env_steps == N * steps
    s = b.stats()
    for p in (moves, rewards, status):
        b.free(p)
    b.close()
    return {"ms_per_tick": ms, "env_steps_per_s": N / (ms * 1e-3), "episodes": s.episodes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=400)
    a = ap.parse_args()
    for game, modes in (("ffa", ("step", "step_generic", "rewards", "rewards_status")),
                        ("teams", ("step", "rewards", "rewards_status"))):
        runs = {m: [] for m in modes}
        for _ in range(a.rounds):
            for m in modes:
                runs[m].append(run(game, m, a.steps))
        gpu = gpu_info()
        for m in modes:
            rates = sorted(r["env_steps_per_s"] for r in runs[m])
            print(json.dumps({"game": game, "mode": m, "env_steps_per_s": rates[len(rates) // 2], "rounds": runs[m],
                              "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
