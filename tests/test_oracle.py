"""CPU tests (-m "not gpu"): pin the oracle.

* the plain-C restatement passes the reference's own known-answer scenarios (tests/scenarios.py);
* it reproduces every golden vector produced by the compiled reference (tests/golden/*.npz);
* where the compiled reference is available (oracle/_ref, build container) the restatement is
  compared with it field by field on fresh random traces, including the kick/bomb stress regime.
"""
import os

import numpy as np
import pytest

import oracle
import scenarios

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("fn", scenarios.STEP_SCENARIOS + scenarios.UTIL_SCENARIOS, ids=lambda f: f.__name__)
def test_scenarios_restatement(orc, fn):
    fn(orc)


@pytest.mark.parametrize("fn", scenarios.STEP_SCENARIOS + scenarios.UTIL_SCENARIOS, ids=lambda f: f.__name__)
def test_scenarios_reference(ref, fn):
    fn(ref)


def test_zero_state_matches_reference(orc, ref):
    assert orc.diff_batch(orc.zero_state(3), ref.zero_state(3))[0] == -1


def test_golden_scenarios(orc):
    g = np.load(os.path.join(GOLD, "scenarios.npz"))
    before = g["before"].copy().view(oracle.STATE_DT).reshape(-1)
    after = g["after"].copy().view(oracle.STATE_DT).reshape(-1)
    moves = g["moves"]
    S = before.copy()
    orc.step_batch(S, np.ascontiguousarray(moves))
    e, why = orc.diff_batch(S, after)
    assert e == -1, "transition %d (%s) differs in field group %d" % (e, g["names"][e], why)


def test_golden_init(orc):
    g = np.load(os.path.join(GOLD, "init.npz"))
    for seed, board in zip(g["seeds"], g["boards"]):
        s = orc.zero_state()
        assert orc.init_board_items(s, int(seed)) == 0
        assert (s["board"][0] == board).all(), hex(int(seed))
    # the default seed is clean, 0x13327 is not (SURVEY §8c D2)
    assert int(g["seeds"][0]) == 0x1337
    assert orc.init_board_items(orc.zero_state(), 0x13327) == 1


@pytest.mark.parametrize("name", ["random6", "harmless5", "stress6"])
def test_golden_traces(orc, name):
    g = np.load(os.path.join(GOLD, "traces.npz"))
    n, ticks, nact, stress, rs = [int(v) for v in g[name + "_cfg"]]
    S = g[name + "_init"].copy().view(oracle.STATE_DT).reshape(-1)
    status = np.zeros(n, np.uint8)
    excluded = g[name + "_excluded"]
    for t in range(ticks):
        mv = orc.rng_moves(rs, 0, n, t, nact)
        live = (excluded < 0) | (excluded > t)
        orc.env_step_batch(S, status, mv)
        h = orc.hash_batch(S)
        bad = (h != g[name + "_hash"][t]) & live
        assert not bad.any(), "tick %d env %d" % (t, int(np.nonzero(bad)[0][0]))
        assert (((status ^ g[name + "_status"][t]) & 0x0F)[live] == 0).all()
    final = g[name + "_final"].copy().view(oracle.STATE_DT).reshape(-1)
    assert orc.diff_batch(S, final, (excluded >= 0).astype(np.uint8))[0] == -1


def test_defect_d5_unbounded_chain_reversion_is_fenced(orc):
    """Found by this project's differential runs: AgentBombChainReversion (step_utility.cpp:89-92) recurses
    forever when the chain reaches an agent whose move is BOMB/IDLE.  Agent 2 plants into a ring slot whose
    stale direction bits say UP (SURVEY Q4), agent 1 kicks a stacked bomb and is bounced back onto the cell
    that stale bomb "moves" to.  The compiled reference hangs (-O3) / overflows its stack (-O0) on this state
    (verified in a forked child in the build container); the restatement flags it and freezes the env."""
    s = np.load(os.path.join(GOLD, "d5_state.npy")).view(oracle.STATE_DT).copy()
    mv = np.array([0, 1, 5, 3], np.uint8)
    st = np.zeros(1, np.uint8)
    fl = np.zeros(1, np.uint8)
    orc.env_step_batch(s, st, mv.reshape(1, 4), fl)
    assert fl[0] & 0x20 and st[0] & 0x10
    before = s.copy()
    orc.env_step_batch(s, st, mv.reshape(1, 4), fl)      # frozen from now on
    assert orc.diff_batch(s, before)[0] == -1 and fl[0] == 0


def test_defect_d5_hangs_the_compiled_reference(ref):
    import signal
    s = np.load(os.path.join(GOLD, "d5_state.npy")).view(oracle.STATE_DT).copy()
    mv = np.array([0, 1, 5, 3], np.uint8)
    assert ref.precheck(s, mv) == 0                      # not predictable by the cheap pre-check
    pid = os.fork()
    if pid == 0:
        signal.alarm(2)
        ref.step(s, mv)
        os._exit(0)
    _, rc = os.waitpid(pid, 0)
    assert rc != 0, "the reference returned from a tick this project believes to be unbounded"


def test_rng_moves_range(orc):
    m6 = orc.rng_moves(7, 0, 4096, 3, 6)
    m5 = orc.rng_moves(7, 0, 4096, 3, 5)
    assert m6.max() == 5 and m5.max() == 4
    # stateless: same (seed, env, tick) -> same moves, different tick -> different stream
    assert (orc.rng_moves(7, 100, 16, 3, 6) == m6[100:116]).all()
    assert (orc.rng_moves(7, 0, 4096, 4, 6) != m6).any()
    counts = np.bincount(m6.reshape(-1), minlength=6)
    assert counts.min() > 4096 * 4 / 6 * 0.9


def _differential(orc, ref, n, ticks, nact, stress, seed):
    seeds = oracle.clean_seeds(128)
    A = ref.zero_state(n)
    B = orc.zero_state(n)
    for e in range(n):
        ref.init_state(A[e:e + 1], seeds[e % len(seeds)])
        assert orc.init_state(B[e:e + 1], seeds[e % len(seeds)]) == 0
    if stress:
        for X in (A, B):
            X["agents"]["canKick"] = 1
            X["agents"]["maxBombCount"] = 5
            X["agents"]["bombStrength"] = 4
    A0, B0 = A.copy(), B.copy()
    sa = np.zeros(n, np.uint8)
    sb = np.zeros(n, np.uint8)
    pre = np.zeros(n, np.uint8)
    fo = np.zeros(n, np.uint8)
    steps = 0
    for t in range(ticks):
        mv = orc.rng_moves(seed, 0, n, t, nact)
        orc.env_step_batch(B, sb, mv, fo)
        # D5 (the reference hangs) can only be detected by running the tick: exclude those envs for the reference
        ref.env_step_batch(A, sa, mv, pre, ((fo & 0x20) != 0).astype(np.uint8))
        skip = ((sa & 0x10) != 0).astype(np.uint8)
        e, why = orc.diff_batch(A, B, skip)
        assert e == -1, "tick %d env %d field group %d" % (t, e, why)
        assert ((((sa ^ sb) & 0x0F) != 0) & (skip == 0)).sum() == 0
        fin = ((sa & 0x11) != 0)
        steps += int((~fin).sum())
        idx = np.nonzero(fin)[0]          # restart finished / excluded envs to keep the traffic up
        A[idx] = A0[idx]
        B[idx] = B0[idx]
        sa[idx] = 0
        sb[idx] = 0
    return steps


def test_differential_random(orc, ref):
    assert _differential(orc, ref, 2048, 100, 6, 0, 1001) > 150000


def test_differential_harmless(orc, ref):
    assert _differential(orc, ref, 1024, 200, 5, 0, 1002) > 150000


def test_differential_stress(orc, ref):
    assert _differential(orc, ref, 2048, 200, 6, 1, 1003) > 300000


@pytest.mark.slow
def test_differential_twenty_million_steps(orc, ref):
    """the long differential behind DESIGN §0's figure, committed: >= 2 x 10^7 env-steps of restatement vs the compiled
    reference, every field after every tick, over the three regimes (random, harmless, all-kick stress)"""
    total = 0
    total += _differential(orc, ref, 32768, 240, 6, 0, 5001)
    total += _differential(orc, ref, 16384, 400, 5, 0, 5002)
    total += _differential(orc, ref, 32768, 260, 6, 1, 5003)
    assert total >= 20_000_000, total


def test_defect_d1_three_on_one_is_canonical_and_fenced(orc):
    """Three agents converge on one occupied cell: two agents are unreachable in the dependency walk and the
    reference continues with i = dependency[-1] (a stack word; -O0 segfaults, -O3 returns a non-canonical board).
    The restatement's canonical result: unreachable agents do not move.  ref_precheck reports 2 (checked where the
    compiled reference is available)."""
    s = orc.zero_state()
    for i, (x, y) in enumerate([(1, 1), (0, 1), (3, 1), (2, 1)]):
        orc.put_agent(s, x, y, i)
    mv = [4, 4, 3, 0]                       # a0 -> a3's cell, a1 -> a0's cell, a2 -> a3's cell, a3 idle
    if oracle.have_reference():
        assert oracle.reference().precheck(s, mv) & 7 == 2
    f = orc.step(s, mv)
    assert f & 1
    for i, (x, y) in enumerate([(1, 1), (0, 1), (3, 1), (2, 1)]):
        scenarios.require_agent(s, i, x, y)


def read_pomtrc(path):
    """POMTRC1 trace file (pomcpp_b200/host/pom_trace.hpp)."""
    import struct
    raw = open(path, "rb").read()
    assert raw[:8] == b"POMTRC1\0"
    n, ticks, flags, _ = struct.unpack("<4I", raw[8:24])
    o = 24
    init = np.frombuffer(raw, oracle.STATE_DT, n, o).copy(); o += n * 1004
    moves = np.frombuffer(raw, np.uint8, ticks * n * 4, o).reshape(ticks, n, 4).copy(); o += ticks * n * 4
    hashes = np.frombuffer(raw, np.uint64, n, o).copy(); o += 8 * n
    status = np.frombuffer(raw, np.uint8, n, o).copy(); o += n
    assert o == len(raw)
    return init, moves, hashes, status, flags


def test_golden_trace_file(orc):
    """The on-disk golden trace (written from the compiled reference) replays bit-exactly on the restatement."""
    init, moves, hashes, status, flags = read_pomtrc(os.path.join(GOLD, "stress96.pomtrc"))
    S = init.copy()
    st = np.zeros(S.shape[0], np.uint8)
    for t in range(moves.shape[0]):
        orc.env_step_batch(S, st, np.ascontiguousarray(moves[t]))
    assert (orc.hash_batch(S) == hashes).all()
    assert (((st ^ status) & 0x1F) == 0).all()
