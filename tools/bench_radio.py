"""Cost of the team radio (pom_batch_step_radio, POM_INIT_RADIO) on one GPU; prints one JSON line per measurement.

    python tools/bench_radio.py [--rounds R] [--steps K]

1 Mi team envs, four uniform random agents, AUTORESET | COUNT, one launch per tick, moves from a ring of 256 sets
pre-generated on the device, uniform random message bytes from a ring of 16 sets, rewards to a device buffer.
  step     rewards       pom_batch_step_rewards on a team handle (the REWARDS image the RADIO image extends)
           radio         pom_batch_step_radio with rewards on a radio handle: 4 message bytes more per env-step
  observe  team          pom_batch_observe_planes (agents 0..3, view 4) on a team handle
           radio         the same on a radio handle (the RADIO image of k_observe_planes)
The record array (1 Mi x 292 B = 306 MB) is larger than the 126 MB L2, so no flush is needed between timed passes.  The
two modes of a measurement are timed in turn, round after round, so that other load on the machine falls on both alike;
each line carries every round's figure and their median, and the card's name, power limit and SM clock read in the run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pomcpp_b200 as pb  # noqa: E402

SEED = 20240229
N = 1 << 20
RING = 256
MSG_RING = 16
OBS_PASSES = 20


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


def run_step(mode, steps):
    b = pb.Batch(N, n_templates=4096, max_ticks=800, teams=True, radio=mode == "radio")
    moves, msgs = b.alloc(4 * N * RING), b.alloc(4 * N * MSG_RING)
    rewards = b.alloc(4 * N)
    for t in range(RING):
        b.generate_moves(moves.value + 4 * N * t, SEED, 100000 + t, 6)
    host = np.random.default_rng(SEED).integers(0, 256, 4 * N * MSG_RING, dtype=np.uint8)
    pb._ck(pb.lib().pom_device_copy(b.device, msgs, host.ctypes.data, host.nbytes))
    b.rollout(96, SEED, 0, 0)                              # untimed: the steady-state mix of game phases
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT

    def tick(k):
        mv = moves.value + 4 * N * (k % RING)
        if mode == "radio":
            b.step_radio(mv, msgs.value + 4 * N * (k % MSG_RING), rewards, None, flags)
        else:
            b.step_rewards(mv, rewards, None, flags)
    for w in range(20):
        tick(w)
    b.sync()
    b.clear_stats()
    b.event(0)
    for k in range(steps):
        tick(20 + k)
    b.event(1)
    ms = b.elapsed_ms() / steps
    s = b.stats()
    assert s.env_steps == N * steps
    for p in (moves, msgs, rewards):
        b.free(p)
    b.close()
    return {"ms_per_tick": ms, "env_steps_per_s": N / (ms * 1e-3), "episodes": s.episodes}


def run_observe(mode):
    b = pb.Batch(N, n_templates=4096, max_ticks=800, teams=True, radio=mode == "radio")
    b.rollout(96, SEED, 0, 0)
    if mode == "radio":
        msgs = b.alloc(4 * N)
        moves = b.alloc(4 * N)
        b.generate_moves(moves, SEED, 7, 6)
        host = np.random.default_rng(SEED).integers(0, 256, 4 * N, dtype=np.uint8)
        pb._ck(pb.lib().pom_device_copy(b.device, msgs, host.ctypes.data, host.nbytes))
        b.step_radio(moves, msgs, None, None, pb.STEP_AUTORESET)
        b.free(msgs); b.free(moves)
    stride = int(pb.lib().pom_batch_obs_stride(b.h))
    obs = b.alloc(4 * stride * pb.OBS_BYTES)
    L = pb.lib()
    for _ in range(3):
        assert L.pom_batch_observe_planes(b.h, obs, 15, 4) == 0
    b.sync()
    b.event(0)
    for _ in range(OBS_PASSES):
        assert L.pom_batch_observe_planes(b.h, obs, 15, 4) == 0
    b.event(1)
    ms = b.elapsed_ms() / OBS_PASSES
    b.free(obs)
    b.close()
    return {"ms_per_call": ms, "envs_per_s": N / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=400)
    a = ap.parse_args()
    for what, modes, fn, key in (("step", ("rewards", "radio"), lambda m: run_step(m, a.steps), "env_steps_per_s"),
                                 ("observe", ("team", "radio"), run_observe, "envs_per_s")):
        runs = {m: [] for m in modes}
        for _ in range(a.rounds):
            for m in modes:
                runs[m].append(fn(m))
        gpu = gpu_info()
        for m in modes:
            rates = sorted(r[key] for r in runs[m])
            print(json.dumps({"bench": what, "mode": m, key: rates[len(rates) // 2], "rounds": runs[m], "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
