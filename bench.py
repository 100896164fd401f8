#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched Pommerman step path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR: after the timed steps, rank 0 writes what its timed region computed as .npy files, so that two builds
can be compared output for output (the inputs depend only on the arguments):
  status.npy  float32 [n_envs]              status byte of every env after the last timed step
  states.npy  float64 [DUMP_ENVS, 263]      the full State of a fixed, seeded sample of envs after the last timed step,
                                            every field of include/pom_state.h flattened in declaration order
  stats.npy   float64 [10]                  the episode counters of the warmup + timed steps (pom_batch_stats)

Own arm (default): BASELINE.json configs[2] — 1,048,576 envs per GPU, random joint actions incl. bombs,
kicks and chain explosions, PER-TICK kernel (pom_batch_step, auto-reset on so every env is live on every
tick).  One "step" = one tick over the whole batch = n_envs env-steps per GPU.  Per-tick joint actions are
pre-generated ON the device for a ring of ticks (inputs resident in HBM when the timed region starts);
the 306 MB record array per GPU is larger than the 126 MB L2, so no flush is needed between steps.
K steps are timed with CUDA events on the launching stream, bracketed by a barrier + device sync, MAX
over ranks.

Further keys of the JSON line (each leg carries its own clock samples):
  roofline        k_step_ws against the measured HBM copy peak (and the nominal 8 TB/s), `single_launch` = ticks strictly
                  one after the other
  e2e             the same metric through the C ABI with pinned HOST buffers, every tick: compact I/O
                  (pom_batch_step_compact: uint16 joint actions in, done bits + finished-env list out), two half-batches
                  stepped alternately; `byte_api` = the byte-per-agent API of round 1 (4 B in, 1 B out per env)
  e2e_obs         e2e with the observation planes of one agent written by the same kernel (they stay on the device)
  legs.rollout    configs[3]: fused 800-tick rollout, 524,288 envs per GPU, in-kernel RNG, auto-reset, counters reduced
                  over ranks with one all-reduce
  legs.expand     configs[4]: 4,096 roots x 6^4 joint actions, clone + one Step each
  legs.strong     configs[2] with 1 Mi envs TOTAL split over the N GPUs (strong scaling)
  parity_sampled  every rank replays strided envs of its shard on the oracle (the checker, not the product)
  cpu_baseline    the UNMODIFIED reference (oracle/_ref) on the box's host cores, bounded sample (rank 0, N=1 only);
                  `ref_flags_value` = the same with the reference's own compiler flags (no -O, Makefile:2)

Reference arm (--impl reference): the reference's own CPU Step on all host cores, one step = one tick over the
SAME 1 Mi envs; same metric / unit / config.

Envs are independent: they shard over GPUs with no data-path collective ("scaling": "weak", per-GPU work
fixed); the only collective is the final all-reduce of the episode counters.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 1 << 20
N_TEMPLATES = 4096
MOVE_RING = 256              # distinct pre-generated ticks of joint actions, cycled
PREROLL_TICKS = 96           # untimed fused rollout so the batch is in its steady-state mix
RNG_SEED = 20240229
ALGO_BYTES = 2 * 289 + 4     # SURVEY §8(d): packed state in + out + 4 move bytes per env-step
NOMINAL_HBM_GBS = 8000.0     # north_star's "~8 TB/s"
CPU_SAMPLE_ENVS = 262144
CPU_SAMPLE_TICKS = 96
E2E_STEPS = 600              # a few hundred ticks at least: 50 were a 6 ms measurement (VERDICT r1)
E2E_BYTE_API_STEPS = 200
ROLLOUT_ENVS_PER_GPU = 524288
ROLLOUT_TICKS = 800
EXPAND_ROOTS, EXPAND_FANOUT = 4096, 1296
STRONG_TOTAL = 1 << 20
PARITY_ENVS, PARITY_TICKS = 64, 48
DUMP_ENVS = 16384            # --dump-outputs: 16 Ki sampled States, 34 MB as float64


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while a timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10}
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            self.sample()
            time.sleep(0.005)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


class clocks_during:
    """with clocks_during(gpu) as c: ...timed region...; c.result() afterwards"""

    def __init__(self, index):
        self.s = ClockSampler(index)

    def __enter__(self):
        self.s.start()
        return self

    def __exit__(self, *a):
        self.s.stop_flag = True
        self.s.join()
        if self.s.ok and not self.s.samples:
            self.s.sample()

    def result(self):
        return self.s.result()


def load_profile(name, key):
    """a figure from the committed ncu summaries (profiles/), or None"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name))).get(key)
    except Exception:
        return None


def traffic_per_tick(n):
    """DRAM bytes per tick of n envs from the committed ncu capture of k_step_ws (which stepped envs_per_launch envs)"""
    t, e = load_profile("k_step_ncu_summary_r2f.json", "dram_bytes_per_launch"), load_profile("k_step_ncu_summary_r2f.json", "envs_per_launch")
    return None if not t or not e else float(t) * n / float(e)


def profile_metric(name, metric):
    try:
        v = json.load(open(os.path.join(ROOT, "profiles", name)))["metrics"][metric]["values"][0]
        return float(str(v).replace(",", ""))
    except Exception:
        return None


# --------------------------------------------------------------------------------------------- CPU legs (the checker side)
def cpu_reference_states(n, preroll, flavour=""):
    """Initial states for the CPU legs, built with the reference's own InitState on clean seeds and
    pre-rolled with the reference's Step so the sample is in the steady-state mix."""
    import oracle
    oracle.build()
    R = None
    if oracle.have_reference():
        try:
            R = oracle.reference(flavour)
        except (FileNotFoundError, OSError):
            R = None
    O = oracle.restatement()
    eng = R if R is not None else O
    kind = "reference" if R is not None else "port"
    seeds = oracle.clean_seeds(N_TEMPLATES)
    T = eng.zero_state(N_TEMPLATES)
    for k, sd in enumerate(seeds):
        eng.init_state(T[k:k + 1], sd)
    S = T[np.arange(n) % N_TEMPLATES].copy()
    status = np.zeros(n, np.uint8)
    cores = os.cpu_count() or 1
    if preroll:
        mv = np.stack([O.rng_moves(RNG_SEED, 0, n, t, 6) for t in range(preroll)])
        eng.bench_steps(S, status, mv, cores, T)
    return eng, O, kind, S, status, T, cores


def cpu_baseline_leg():
    eng, O, kind, S, status, T, cores = cpu_reference_states(CPU_SAMPLE_ENVS, 32)
    mv = np.stack([O.rng_moves(RNG_SEED, 0, CPU_SAMPLE_ENVS, 1000 + t, 6) for t in range(CPU_SAMPLE_TICKS)])
    best = 0.0
    for _ in range(2):
        t, steps = eng.bench_steps(S, status, mv, cores, T)
        best = max(best, steps / t)
    out = {"value": best, "unit": "env-steps/s", "cores": cores, "kind": kind,
           "sample": "%d envs x %d ticks (auto-reset), best of 2, reference Step -O3, %d threads" %
                     (CPU_SAMPLE_ENVS, CPU_SAMPLE_TICKS, cores)}
    # the same loop built with the reference's own flags (its Makefile:2 passes no -O): oracle/_ref/libpomref_O0.so
    try:
        import oracle
        if kind == "reference":
            slow = oracle.reference("_O0")
            n0 = CPU_SAMPLE_ENVS // 4
            S0, st0 = S[:n0].copy(), np.zeros(n0, np.uint8)
            t, steps = slow.bench_steps(S0, st0, np.ascontiguousarray(mv[:32, :n0]), cores, T)
            out["ref_flags_value"] = steps / t
            out["ref_flags_sample"] = "%d envs x 32 ticks, reference built with its own flags (-std=c++17 -pthread, no -O)" % n0
    except Exception as e:                                   # the -O0 flavour is optional
        out["ref_flags_value"] = None
        out["ref_flags_sample"] = "unavailable: %s" % e
    return out


def fence_overhead(eng, O, cores):
    """what the reference arm's per-tick defect fence (FenceTick, oracle/ref_shim.cpp) costs: the same Harmless trace -
    no bombs, so the fence can never fire - timed with and without it"""
    if not hasattr(eng, "set_fence"):
        return None
    n, ticks = 131072, 48
    seeds = __import__("oracle").clean_seeds(256)
    T = eng.zero_state(256)
    for k, sd in enumerate(seeds):
        eng.init_state(T[k:k + 1], sd)
    mv = np.stack([O.rng_moves(RNG_SEED + 1, 0, n, t, 5) for t in range(ticks)])
    res = {}
    for on in (1, 0, 1, 0, 1, 0, 1, 0):
        S = T[np.arange(n) % 256].copy()
        st = np.zeros(n, np.uint8)
        eng.set_fence(on)
        t, steps = eng.bench_steps(S, st, mv, cores, T)
        res[on] = max(res.get(on, 0.0), steps / t)
    eng.set_fence(1)
    return {"with_fence": res[1], "without_fence": res[0], "slowdown": res[0] / res[1] - 1.0,
            "sample": "%d envs x %d Harmless ticks (the cheapest tick there is: the fence weighs most here), best of 4 each" % (n, ticks)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = ENVS_PER_GPU                                    # the own arm's batch: same config
    eng, O, kind, S, status, T, cores = cpu_reference_states(n, 32)
    K, W = args.steps, args.warmup
    ring = np.stack([O.rng_moves(RNG_SEED, 0, n, 2000 + t, 6) for t in range(min(32, K + W))])
    R = ring.shape[0]
    if W:
        eng.bench_steps(S, status, np.ascontiguousarray(ring[np.arange(W) % R]), cores, T)
    # ONE call for the K timed ticks: the threads are spawned once, not per tick
    t, steps = eng.bench_steps(S, status, np.ascontiguousarray(ring[(W + np.arange(K)) % R]), cores, T)
    v = steps / t
    line = {"impl": "reference", "metric": "env-steps/sec", "value": v, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * t / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": "configs[2]: %d envs x 4 random agents (uniform{0..5}: moves, bombs, kicks, chain explosions), "
                                   "auto-reset, reference bboard::Step (-O3) on the host cores; one step = one tick over all envs" % n,
                       "envs_per_step": n, "threads": cores, "same_config": True},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": kind,
                             "sample": "%d envs per step, %d steps in one threaded call" % (n, K)},
            "fence_overhead": fence_overhead(eng, O, cores),
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- own arm
def oracle_replay(O, T, first_env, global_envs, ticks, seed, max_ticks):
    """host replay of the per-tick auto-reset rule for single envs (tests/test_gpu_parity.py::_oracle_rollout)"""
    nT = T.shape[0]
    out_S, out_st = [], []
    for g in global_envs:
        S = T[(g % nT):(g % nT) + 1].copy()
        st = np.zeros(1, np.uint8)
        ep = 0
        for k in range(ticks):
            mv = O.rng_moves(seed, int(g), 1, k, 6)
            O.env_step_batch(S, st, mv)
            if max_ticks and not (st[0] & 1) and S["timeStep"][0] >= max_ticks:
                st[0] |= 0x20
            if st[0] & 0x31:
                ep += 1
                S[0] = T[(g + ep) % nT]
                st[0] = 0
        out_S.append(S)
        out_st.append(st)
    return np.concatenate(out_S), np.concatenate(out_st)


def dump_outputs(pb, b, counters, out_dir):
    """--dump-outputs: the timed region's results on `b` (see the module docstring); call before anything else steps `b`"""
    from numpy.lib import recfunctions
    idx = np.sort(np.random.default_rng(RNG_SEED).choice(b.n, min(DUMP_ENVS, b.n), replace=False)).astype(np.uint32)
    small = pb.Batch(idx.shape[0], device=b.device, n_templates=1, empty=True)
    small.clone_from(b, idx)
    S, _ = small.download()
    small.close()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "status.npy"), b.status().astype(np.float32))
    np.save(os.path.join(out_dir, "states.npy"), recfunctions.structured_to_unstructured(S, dtype=np.float64))
    np.save(os.path.join(out_dir, "stats.npy"), counters.astype(np.float64))


def run_own(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    torch = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import pomcpp_b200 as pb
    from pomcpp_b200 import shard
    pb.bind_thread_near(local_rank)                    # this rank's host thread next to its GPU (launches, polling)
    n = ENVS_PER_GPU
    K, W = args.steps, args.warmup
    plan = shard.shard_plan(rank, world, n)
    b = pb.Batch(n, device=local_rank, env_offset=plan["first"], n_templates=N_TEMPLATES, max_ticks=800)
    ring = min(MOVE_RING, K + W)
    moves_dev = b.alloc(4 * n * ring)
    for t in range(ring):
        b.generate_moves(moves_dev.value + 4 * n * t, RNG_SEED, 100000 + t, 6)
    b.rollout(PREROLL_TICKS, RNG_SEED, 0, 0)          # untimed: reach the steady-state mix
    b.sync()
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT
    dev = "cuda" if dist is not None else "cpu"

    def barrier(*handles):
        for h in handles or (b,):
            h.sync()
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier()

    # ---- the kernel alone: one launch per tick over the whole batch, ticks strictly one after the other
    SINGLE_STEPS = min(200, K)
    for w in range(5):
        b.step(moves_dev.value + 4 * n * (w % ring), flags)
    b.sync()
    b.event(0)
    for k in range(SINGLE_STEPS):
        b.step(moves_dev.value + 4 * n * (k % ring), flags)
    b.event(1)
    single_ms = b.elapsed_ms() / SINGLE_STEPS
    b.sync()
    b.clear_stats()
    # ---- the timed region proper: the same kernel, the two halves of the batch on two streams (POM_STEP_OVERLAP): while
    #      one launch drains, the other fills
    if os.environ.get("POM_BENCH_OVERLAP", "1") != "0":
        flags |= pb.STEP_OVERLAP
    flags_main = flags
    for w in range(W):
        b.step(moves_dev.value + 4 * n * (w % ring), flags)
    barrier()
    with clocks_during(local_rank) as main_clocks:
        l0 = b.launch_count()
        b.event(0)
        for k in range(K):
            b.step(moves_dev.value + 4 * n * ((W + k) % ring), flags)
        b.event(1)
        ms = b.elapsed_ms()
        barrier()
    launches = b.launch_count() - l0
    stats = b.stats()
    assert stats.env_steps == n * (K + W), "kernel did not step every env on every tick"
    counters_main = b.stats().as_array()
    if args.dump_outputs and rank == 0:
        dump_outputs(pb, b, counters_main, args.dump_outputs)
    flags &= ~pb.STEP_OVERLAP

    # ---- e2e: HOST buffers through the C ABI, every tick, the host waits for every result.  The envs run as two
    #      half-batches stepped alternately (an actor loop with two env groups): while the host consumes the results of
    #      one half, the GPU steps the other.  Compact I/O: 2 bytes of joint action per env in; one done bit per env and
    #      the list of finished envs (index + status byte) out.  Pinned buffers live on the GPU's NUMA node.
    h = n // 2
    E2E_RING = 32                                        # distinct move sets: a short ring would make the games periodic
    halves = [pb.Batch(h, device=local_rank, env_offset=plan["first"] + i * h, n_templates=N_TEMPLATES, max_ticks=800) for i in range(2)]
    for x in halves:
        x.rollout(PREROLL_TICKS, RNG_SEED, 0, 0)
        x.sync()
    owners = []

    def pinned(shape, dt):
        arr, o = pb.pinned_array(shape, dt, near_device=local_rank)
        owners.append(o)
        return arr

    rng = np.random.default_rng(RNG_SEED + rank)
    joint = [[pinned((h,), np.uint16) for _ in range(E2E_RING)] for _ in range(2)]
    for i in range(2):
        for arr in joint[i]:
            arr[:] = rng.integers(0, 1296, size=h, dtype=np.uint16)      # the policy's output, already in pinned memory
    bits = [pinned(((h + 31) // 32,), np.uint32) for _ in range(2)]
    fenv = [pinned((h,), np.uint32) for _ in range(2)]
    fst = [pinned((h,), np.uint8) for _ in range(2)]
    fcnt = [pinned((1,), np.uint32) for _ in range(2)]
    obs_dev = [None, None]

    def compact_loop(steps, with_obs):
        fin_total = 0
        # the I/O descriptors are built once: an actor loop reuses its buffers
        ios = [[halves[i].compact_io(joint[i][k], bits[i], fenv[i], fst[i], fcnt[i],
                                     obs_dev[i] if with_obs else None, 1 if with_obs else 0, 4) for k in range(E2E_RING)] for i in range(2)]

        def go(i, k):
            halves[i].step_compact_io(ios[i][k % E2E_RING], flags)
        go(0, 0)
        for k in range(steps):
            go(1, k)
            halves[0].sync()                   # results of half 0 are on the host now; its next actions are read from here
            fin_total += int(fcnt[0][0])
            if k + 1 < steps:
                go(0, k + 1)
            halves[1].sync()
            fin_total += int(fcnt[1][0])
        return fin_total

    compact_loop(8, False)
    barrier(*halves)
    with clocks_during(local_rank) as e2e_clocks:
        t0 = time.perf_counter()
        fin_seen = compact_loop(E2E_STEPS, False)
        e2e_s = time.perf_counter() - t0
        barrier(*halves)
    d2h_compact = 2 * (4 * ((h + 31) // 32) + 4) + 5.0 * fin_seen / E2E_STEPS      # bits + count words + list entries, per tick

    # e2e with the observation planes of agent 0 (view 4) written by the step kernel; they stay on the device, where a
    # policy network would read them
    stride = int(pb.lib().pom_batch_obs_stride(halves[0].h))
    for i in range(2):
        obs_dev[i] = halves[i].alloc(stride * pb.OBS_BYTES)
    compact_loop(8, True)
    barrier(*halves)
    with clocks_during(local_rank) as obs_clocks:
        t0 = time.perf_counter()
        compact_loop(E2E_STEPS // 2, True)
        e2e_obs_s = time.perf_counter() - t0
        barrier(*halves)
    for i in range(2):
        halves[i].free(obs_dev[i])

    # the byte-per-agent API of round 1 on the same halves (4 move bytes in, 1 status byte out per env)
    mv4 = [[pinned((h, 4), np.uint8) for _ in range(4)] for _ in range(2)]
    st1 = [pinned((h,), np.uint8) for _ in range(2)]
    for i in range(2):
        for arr in mv4[i]:
            arr[:] = rng.integers(0, 6, size=(h, 4), dtype=np.uint8)

    def byte_loop(steps):
        halves[0].step_host_async(mv4[0][0], st1[0], flags)
        for k in range(steps):
            halves[1].step_host_async(mv4[1][k % 4], st1[1], flags)
            halves[0].sync()
            if k + 1 < steps:
                halves[0].step_host_async(mv4[0][(k + 1) % 4], st1[0], flags)
            halves[1].sync()

    byte_loop(8)
    barrier(*halves)
    t0 = time.perf_counter()
    byte_loop(E2E_BYTE_API_STEPS)
    e2e_byte_s = time.perf_counter() - t0
    barrier(*halves)
    e2e_launches = halves[0].launch_count() + halves[1].launch_count()
    for x in halves:
        x.close()
    # one batch, synchronous call per tick (pom_batch_step_host): launch and wait
    mvw, stw = pinned((n, 4), np.uint8), pinned((n,), np.uint8)
    mvw[:] = rng.integers(0, 6, size=(n, 4), dtype=np.uint8)
    for w in range(5):
        b.step_host(mvw, stw, flags)
    barrier()
    t0 = time.perf_counter()
    for k in range(100):
        b.step_host(mvw, stw, flags)
    e2e_single_s = (time.perf_counter() - t0) / 100 * E2E_STEPS
    barrier()

    # ---- legs.rollout: configs[3], fused 800-tick rollout with in-kernel RNG and auto-reset
    rb = pb.Batch(ROLLOUT_ENVS_PER_GPU, device=local_rank, env_offset=rank * ROLLOUT_ENVS_PER_GPU, n_templates=N_TEMPLATES, max_ticks=800)
    rb.rollout(64, RNG_SEED, 0, 0)
    rb.clear_stats()
    barrier(rb)
    with clocks_during(local_rank) as roll_clocks:
        rb.event(0)
        rb.rollout(ROLLOUT_TICKS, RNG_SEED, 64, 0)
        rb.event(1)
        roll_ms = rb.elapsed_ms()
        barrier(rb)
    roll_counters = rb.stats().as_array()
    assert int(roll_counters[0]) == ROLLOUT_ENVS_PER_GPU * ROLLOUT_TICKS
    rb.close()

    # ---- legs.expand: configs[4], 4096 roots x 6^4 joint actions, clone + one Step each (one kernel)
    eb = pb.Batch(EXPAND_ROOTS * EXPAND_FANOUT, device=local_rank, n_templates=16, empty=True)
    roots = (np.arange(EXPAND_ROOTS, dtype=np.uint32) * 251) % n      # roots: mid-game states of the main batch
    eb.expand_step_from(b, roots, EXPAND_FANOUT, 0)
    barrier(eb)
    with clocks_during(local_rank) as exp_clocks:
        EXP_REPS = 10
        eb.event(0)
        for _ in range(EXP_REPS):
            eb.expand_step_from(b, roots, EXPAND_FANOUT, 0)           # enqueues: index upload + one kernel
        eb.event(1)
        exp_s = eb.elapsed_ms() / 1e3 / EXP_REPS
        barrier(eb)
    eb.close()

    # ---- roofline.big_batch: the same kernel on 4 Mi envs per GPU (1.2 GB of records): a launch's fill and drain
    #      (about 10 us: the first loads before any store, the last slices of every CTA) is 10 % of a 1 Mi-env tick
    #      and 2.5 % of this one - what the kernel sustains, as opposed to what one configs[2] tick costs
    BIG = 4 * (1 << 20)
    bb = pb.Batch(BIG, device=local_rank, env_offset=plan["first"] * 4, n_templates=N_TEMPLATES, max_ticks=800)
    bb.rollout(PREROLL_TICKS, RNG_SEED, 0, 0)
    big_ring = 6
    big_moves = bb.alloc(4 * BIG * big_ring)
    for t in range(big_ring):
        bb.generate_moves(big_moves.value + 4 * BIG * t, RNG_SEED, 200000 + t, 6)
    big_flags = flags_main            # as in the timed region (POM_STEP_OVERLAP unless POM_BENCH_OVERLAP=0)
    for w in range(4):
        bb.step(big_moves.value + 4 * BIG * (w % big_ring), big_flags)
    barrier(bb)
    BIG_STEPS = 20
    bb.event(0)
    for k in range(BIG_STEPS):
        bb.step(big_moves.value + 4 * BIG * (k % big_ring), big_flags)
    bb.event(1)
    big_ms = bb.elapsed_ms() / BIG_STEPS
    barrier(bb)
    bb.free(big_moves)
    bb.close()

    # ---- legs.strong: 1 Mi envs in TOTAL split over the ranks, per-tick kernel
    sp = shard.strong_plan(rank, world, STRONG_TOTAL)
    sb = pb.Batch(sp["count"], device=local_rank, env_offset=sp["first"], n_templates=N_TEMPLATES, max_ticks=800)
    sb.rollout(PREROLL_TICKS, RNG_SEED, 0, 0)
    for w in range(5):
        sb.step(moves_dev.value + 4 * n * (w % ring), flags_main)
    barrier(sb)
    with clocks_during(local_rank) as strong_clocks:
        sb.event(0)
        for k in range(K):
            sb.step(moves_dev.value + 4 * n * (k % ring), flags_main)
        sb.event(1)
        strong_ms = sb.elapsed_ms()
        barrier(sb)
    sb.close()

    # ---- parity_sampled: strided envs of this rank's shard replayed on the oracle from the same templates and the same
    #      stateless action source (keyed by the GLOBAL env index: results must not depend on the GPU count)
    import oracle
    O = oracle.restatement()
    b.reset()
    T, _ = b.templates()
    pm = b.alloc(4 * n)
    for t in range(PARITY_TICKS):
        b.generate_moves(pm, RNG_SEED + 7, t, 6)
        b.step(pm, pb.STEP_AUTORESET)
    b.free(pm)
    local_idx = (np.arange(PARITY_ENVS, dtype=np.uint32) * (n // PARITY_ENVS) + 13 * rank) % n
    small = pb.Batch(PARITY_ENVS, device=local_rank, n_templates=1, empty=True)
    small.clone_from(b, local_idx)
    G, gst = small.download()
    small.close()
    want, wst = oracle_replay(O, T, plan["first"], plan["first"] + local_idx.astype(np.int64), PARITY_TICKS, RNG_SEED + 7, 800)
    mismatches = 0
    for e in range(PARITY_ENVS):
        if O.diff_batch(G[e:e + 1], want[e:e + 1])[0] != -1 or gst[e] != wst[e]:
            mismatches += 1

    # ---- aggregate over ranks
    t_max = [float(v) for v in shard.max_over_ranks([ms, e2e_s, e2e_single_s, e2e_byte_s, e2e_obs_s, roll_ms, exp_s, strong_ms], dist, dev)]
    ms_max, e2e_max, e2e_single_max, e2e_byte_max, e2e_obs_max, roll_max, exp_max, strong_max = t_max
    # the one collective of the run: final reduce of the episode counters (+ the parity mismatches)
    counters = shard.reduce_counters(counters_main, dist, dev)
    roll_total = shard.reduce_counters(roll_counters, dist, dev)
    parity = shard.reduce_counters(np.array([PARITY_ENVS, mismatches, int(d2h_compact)], np.int64), dist, dev)

    if rank == 0:
        peak, peak_src = measured_peak()
        value = world * n * K / (ms_max * 1e-3)
        achieved = ALGO_BYTES * n / (ms / K * 1e-3) / 1e9           # this rank's kernel, GB/s
        single_achieved = ALGO_BYTES * n / (single_ms * 1e-3) / 1e9
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_max / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
            "config": {"workload": "configs[2]: %d envs per GPU x 4 random agents (uniform{0..5}: moves, bombs, kicks, chain "
                                   "explosions), per-tick kernel pom_batch_step (k_step_ws: persistent, one CTA per SM), auto-reset, "
                                   "POM_STEP_OVERLAP (the two halves of the batch on two streams)" % n,
                       "envs_per_gpu": n, "envs_total": world * n, "record_bytes": 292, "templates": N_TEMPLATES,
                       "preroll_ticks": PREROLL_TICKS, "move_ring_ticks": ring,
                       "l2": "record array %d MB per GPU > 126 MB L2: every step streams from HBM, no flush needed" % (n * 292 // 2 ** 20),
                       "parallelism": "env-sharded x%d, no data-path collective" % world},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_nominal_8tbs": achieved / NOMINAL_HBM_GBS,
                         "traffic": traffic_per_tick(n),
                         "algorithmic_bytes_per_env_step": ALGO_BYTES,
                         "peak_source": peak_src, "kernel": "k_step_ws<20,24>", "step_ms": ms / K,
                         "launches_per_step": 2,
                         "note": "achieved = 582 B x envs / time per tick over the timed region (CUDA events bracket both streams); traffic = DRAM "
                                 "bytes per tick, scaled from the ncu capture of one half-batch launch (profiles/k_step_ncu_summary_r2f.json)",
                         "big_batch": {"envs_per_gpu": 4 * (1 << 20), "launch_ms": big_ms, "achieved": ALGO_BYTES * 4 * (1 << 20) / (big_ms * 1e-3) / 1e9,
                                       "frac": ALGO_BYTES * 4 * (1 << 20) / (big_ms * 1e-3) / 1e9 / peak, "steps": 20,
                                       "what": "the timed region's call on 4 Mi envs per GPU: the per-launch fill and drain amortised (this rank)"},
                         "single_launch": {"launch_ms": single_ms, "achieved": single_achieved, "frac": single_achieved / peak,
                                           "frac_nominal_8tbs": single_achieved / NOMINAL_HBM_GBS, "steps": SINGLE_STEPS,
                                           "what": "one launch per tick over the whole batch, no overlap between ticks"}},
            "e2e": {"value": world * n * E2E_STEPS / e2e_max, "unit": "env-steps/s",
                    "h2d_bytes_per_step": 2 * n, "d2h_bytes_per_step": int(parity[2] // world), "steps": E2E_STEPS,
                    "clocks": e2e_clocks.result(),
                    "api": "pom_batch_step_compact on two half-batches stepped alternately: pinned host buffers on the GPU's NUMA node; "
                           "per env a uint16 joint action in; a done bit per env plus the list of finished envs (index, status) out; "
                           "the host waits for every half-batch every tick; the kernel reads / writes the host buffers itself",
                    "byte_api": {"value": world * n * E2E_BYTE_API_STEPS / e2e_byte_max, "unit": "env-steps/s",
                                 "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": n, "steps": E2E_BYTE_API_STEPS,
                                 "api": "pom_batch_step_host_async, 4 move bytes in and 1 status byte out per env (round 1's e2e)"},
                    "single_batch": {"value": world * n * E2E_STEPS / e2e_single_max, "unit": "env-steps/s", "steps": 100,
                                     "api": "one batch, pom_batch_step_host: launch and wait, tick after tick"}},
            "e2e_obs": {"value": world * n * (E2E_STEPS // 2) / e2e_obs_max, "unit": "env-steps/s", "steps": E2E_STEPS // 2,
                        "ms_per_1Mi_env_steps": 1e3 * e2e_obs_max / (E2E_STEPS // 2) * (1 << 20) / n,
                        "clocks": obs_clocks.result(),
                        "api": "the e2e loop with obs_dev set: every step also leaves agent 0's observation planes (view 4, 512 B per env) on "
                               "the device, where a policy network would read them (k_observe_planes queued behind the step kernel by the "
                               "same call; POM_OBS_FUSED=1 selects the fused kernel, which is slower)"},
            "legs": {
                "rollout": {"value": float(roll_total[0]) / (roll_max * 1e-3), "unit": "env-steps/s", "ms": roll_max,
                            "envs_per_gpu": ROLLOUT_ENVS_PER_GPU, "ticks": ROLLOUT_TICKS,
                            "what": "configs[3]: fused %d-tick rollout, in-kernel counter RNG, auto-reset, counters all-reduced" % ROLLOUT_TICKS,
                            "episodes": int(roll_total[1]), "wins": [int(x) for x in roll_total[2:6]], "draws": int(roll_total[6]),
                            "invalid": int(roll_total[9]),
                            "issue_slot_pct": profile_metric("k_rollout_ncu_summary_r2f.json", "smsp__issue_active.avg.pct_of_peak_sustained_active"),
                            "smem_wavefront_pct": profile_metric("k_rollout_ncu_summary_r2f.json", "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"),
                            "clocks": roll_clocks.result()},
                "expand": {"value": world * EXPAND_ROOTS * EXPAND_FANOUT / exp_max, "unit": "children/s", "ms": 1e3 * exp_max,
                           "roots": EXPAND_ROOTS, "fanout": EXPAND_FANOUT,
                           "write_gbs": EXPAND_ROOTS * EXPAND_FANOUT * 289 / exp_max / 1e9,
                           "write_frac_of_peak": EXPAND_ROOTS * EXPAND_FANOUT * 289 / exp_max / 1e9 / peak,
                           "what": "configs[4]: pom_batch_expand_step, clone + one Step per child in one kernel; CUDA events around 10 calls "
                                   "back to back, incl. the upload of the root index array", "clocks": exp_clocks.result()},
                "strong": {"value": STRONG_TOTAL * K / (strong_max * 1e-3), "unit": "env-steps/s", "ms_per_step": strong_max / K,
                           "envs_total": STRONG_TOTAL, "envs_per_gpu": STRONG_TOTAL // world, "scaling": "strong",
                           "what": "configs[2] with 1 Mi envs in total split over the GPUs, the timed region's call (pom_batch_step with POM_STEP_OVERLAP; it applies from 0.25 Mi envs per GPU up)",
                           "clocks": strong_clocks.result()}},
            "parity_sampled": {"envs": int(parity[0]), "ticks": PARITY_TICKS, "mismatches": int(parity[1]),
                               "what": "every rank: strided envs of its shard after %d per-tick auto-reset steps vs the oracle's replay "
                                       "from the same templates and global-env-keyed actions; every field + status" % PARITY_TICKS},
            "gpu_launches": int(launches),
            "clocks": main_clocks.result(),
            "episode_stats": {"env_steps": int(counters[0]), "episodes": int(counters[1]),
                              "wins": [int(x) for x in counters[2:6]], "draws": int(counters[6]),
                              "truncated": int(counters[7]), "sum_episode_len": int(counters[8]),
                              "invalid": int(counters[9]), "reduced_with": "nccl all_reduce" if world > 1 else "single rank"},
        }
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_leg()
        print(json.dumps(line), flush=True)

    for o in owners:
        pb.pinned_free(o)
    b.free(moves_dev)
    b.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and int(parity[1]) != 0:
        sys.exit("parity_sampled: %d sampled envs differ from the oracle" % int(parity[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed region's results to DIR/*.npy (own arm; with several GPUs, rank 0's shard)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs applies to the own arm")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
