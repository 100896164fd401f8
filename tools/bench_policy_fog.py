"""Throughput of the device SimpleAgent under fog of war (pom_batch_set_policy_view) against the full-state agent on one
GPU; prints one JSON line per leg and mode and appends them to --out.

    python tools/bench_policy_fog.py [--rounds R] [--ticks K] [--out profiles/bench_policy_fog.jsonl]

 rollout      four SimpleAgents per env through pom_batch_rollout(ROLL_SIMPLE(15)) at 1 Mi envs: the default path for
              that size, k_policy_moves + the per-tick step kernel, tick by tick; auto-reset, 800-tick limit
 moves_step   the same game driven by the caller: pom_batch_policy_moves (mask 15) into a device buffer, then pom_batch_step
              with AUTORESET | COUNT, every tick
 modes        ffa_full, ffa_view4, team_full, team_view4 (view 4 = Pommerman's competition setting)

Every handle first plays 40 untimed ticks, so that the games have developed and the policy memories exist; then K ticks
are timed with CUDA events.  1 Mi records are 306 MB, more than the 126 MB L2, so no flush is needed between passes.  The
modes of a leg are timed in turn, round after round, so that other load on the machine falls on all of them alike; each
line carries every round's figure and their median, with the card's name, power limit and clocks read in the same run.
The episode counters show how the fog changes the games themselves (fogged agents neither hunt nor flee what they do not
see, so episodes last differently), which is part of what the figures compare.
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
WARM = 40
MODES = {"ffa_full": (False, -1), "ffa_view4": (False, 4), "team_full": (True, -1), "team_view4": (True, 4)}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


def make(mode):
    teams, view = MODES[mode]
    b = pb.Batch(N, n_templates=4096, max_ticks=800, teams=teams)
    b.set_policy_view(view)
    return b


def counters(b):
    s = b.stats()
    return {"episodes": s.episodes, "mean_episode_len": s.sum_episode_len / max(1, s.episodes), "wins": list(s.wins),
            "draws": s.draws, "truncated": s.truncated, "invalid": s.invalid}


def rollout_leg(mode, ticks):
    b = make(mode)
    b.rollout(WARM, SEED, 0, pb.ROLL_SIMPLE(15))
    b.sync()
    b.clear_stats()
    b.event(0)
    b.rollout(ticks, SEED, WARM, pb.ROLL_SIMPLE(15))
    b.event(1)
    ms = b.elapsed_ms()
    c = counters(b)
    b.close()
    return {"ms": ms, "env_steps_per_s": N * ticks / (ms * 1e-3), **c}


def moves_step_leg(mode, ticks):
    b = make(mode)
    mv = b.alloc(4 * N)
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT
    for t in range(WARM):
        b.policy_moves(mv, SEED, t, 15)
        b.step(mv, flags)
    b.sync()
    b.clear_stats()
    b.event(0)
    for t in range(WARM, WARM + ticks):
        b.policy_moves(mv, SEED, t, 15)
        b.step(mv, flags)
    b.event(1)
    ms = b.elapsed_ms()
    c = counters(b)
    b.free(mv)
    b.close()
    return {"ms": ms, "env_steps_per_s": N * ticks / (ms * 1e-3), **c}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--out", default=None, help="JSON-lines file the results are appended to")
    a = ap.parse_args()
    gpu = gpu_info()
    lines = []
    for leg, fn in (("rollout", rollout_leg), ("moves_step", moves_step_leg)):
        runs = {m: [] for m in MODES}
        for _ in range(a.rounds):
            for m in MODES:
                runs[m].append(fn(m, a.ticks))
        for m in MODES:
            rates = sorted(r["env_steps_per_s"] for r in runs[m])
            line = json.dumps({"leg": leg, "mode": m, "envs": N, "ticks": a.ticks, "env_steps_per_s": rates[len(rates) // 2],
                               "rounds": runs[m], "gpu": gpu})
            print(line, flush=True)
            lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
