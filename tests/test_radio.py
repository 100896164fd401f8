"""Pommerman's team radio (POM_INIT_RADIO, pom_batch_step_radio).  The reference has no radio, so this file holds the
definition, after Pommerman's team-radio environment (pommerman/envs/v2.py), and pins the device code to it:
  RadioRestatement   TeamRestatement plus a [n, 4] array of last messages (w0 | w1 << 3 per agent).  Per env and tick:
                       not stepped (DONE or INVALID when the tick starts)  the messages stay
                       stepped   agent a's message <- msgs[a] & 63 if a was alive when the tick started, else (0, 0)
                       the env ended and is auto-reset                     (0, 0) for everyone
                     Every other call leaves the messages of running envs alone; (re-)initialisation clears them.
  radio_planes       the observation planes of the oracle (pom_oracle_observe_planes / _cropped) with the teammate's
                     (a ^ 2) last message in bytes 493, 494 (full layout) or 4 W^2 + 9, 4 W^2 + 10 (cropped layout).
  CPU  tests/radiosim (pomcore::radio_latch, the team tick, truncation, auto-reset and tick_rewards as k_step_ws runs
       them; observe_planes<RADIO>) == the restatement on random, harmless, stress and inconsistent states, on explicit
       cases, and in both layouts at views 0..5.
  GPU  pom_batch_step_radio on radio handles of 4099 envs == the restatement on every tick, bit-identical in states,
       status bytes, counters and rewards to a twin non-radio team handle driven by pom_batch_step_rewards; every other
       entry point leaves messages alone or clears them on reset; the unfused step_observe; the refusals;
       bboard::BatchEnvironment::StepRadio and GetMessage."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_rewards import reward_definition
from test_teams import TeamRestatement, _games

DONE, DRAW, INVALID, TRUNC = 0x01, 0x02, 0x10, 0x20
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def radio_planes(orc, S, M, agent, view, cropped=False):
    """the observation of `agent` on a radio handle: the oracle's planes plus the teammate's words"""
    if cropped:
        out = orc.observe_cropped_batch(S, agent, view)
        at = 4 * (2 * view + 1) ** 2 + 9
    else:
        out = orc.observe_planes_batch(S, agent, view)
        at = 493
    mate = np.asarray(M)[:, agent ^ 2]
    out[:, at] = mate & 7
    out[:, at + 1] = (mate >> 3) & 7
    return out


class RadioRestatement:
    """TeamRestatement replaying pom_batch_step_radio: the radio rule, Environment::Step with the team rule, truncation at
    max_ticks and reset to template[(env_offset + e + episode) % n_templates] when auto-resetting.  tick() returns the
    status bytes before the reset and the rewards (the status-byte form of tests/test_rewards.py)."""

    def __init__(self, orc, S, T, env0=0, max_ticks=0, autoreset=True):
        self.game = TeamRestatement(orc)
        self.S, self.T, self.env0, self.autoreset = S, T, env0, autoreset
        self.max_ticks = max_ticks if autoreset else 0
        n = S.shape[0]
        self.status = np.zeros(n, np.uint8)
        self.episode = np.zeros(n, np.int64)
        self.M = np.zeros((n, 4), np.uint8)

    def tick(self, mv, msgs):
        S, st = self.S, self.status
        stepped = (st & (DONE | INVALID)) == 0
        alive = S["agents"]["dead"] == 0                      # at the start of the tick
        self.M[stepped] = np.where(alive[stepped], np.asarray(msgs)[stepped] & 63, 0)
        self.game.env_step_batch(S, st, np.ascontiguousarray(mv))
        if self.max_ticks:
            st[stepped & ((st & DONE) == 0) & (S["timeStep"] >= self.max_ticks)] |= TRUNC
        end = st.copy()
        want = reward_definition(stepped, end, S["agents"]["dead"] != 0, True)
        if self.autoreset:
            for e in np.nonzero(stepped & ((end & (DONE | INVALID | TRUNC)) != 0))[0]:
                self.episode[e] += 1
                S[e] = self.T[(self.env0 + e + self.episode[e]) % self.T.shape[0]]
                st[e] = 0
                self.M[e] = 0
        return end, want


class RadioSim:
    """tests/radiosim on packed records (packed by tests/hostsim)"""

    def __init__(self, so, templates=None, env0=0, max_ticks=0, autoreset=True):
        from hostsim import HostSim
        self.h = HostSim()
        L = self.lib = C.CDLL(so)
        vp = C.c_void_p
        L.radiosim_tick.argtypes = [vp, C.c_long, vp, vp, C.c_int, C.c_uint32, vp, C.c_long, C.c_uint64, vp, vp, vp]
        L.radiosim_messages.argtypes = [vp, C.c_long, vp]
        L.radiosim_observe.argtypes = [vp, C.c_long, C.c_int, C.c_int, C.c_int, vp]
        L.radiosim_init_record_radio.argtypes = [C.c_int, vp]
        self.env0, self.max_ticks, self.autoreset = env0, max_ticks, autoreset
        self.tmpl = self.h.pack(templates)[0] if templates is not None else np.zeros((1, 292), np.uint8)

    def tick(self, recs, episodes, mv, msgs):
        n = recs.shape[0]
        st, rw = np.zeros(n, np.uint8), np.zeros((n, 4), np.int8)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.radiosim_tick(p(recs), n, p(np.ascontiguousarray(mv)), p(np.ascontiguousarray(msgs, dtype=np.uint8)),
                               int(self.autoreset), self.max_ticks, p(self.tmpl), self.tmpl.shape[0], self.env0, p(episodes),
                               p(st), p(rw))
        return st, rw

    def messages(self, recs):
        out = np.zeros((recs.shape[0], 4), np.uint8)
        self.lib.radiosim_messages(recs.ctypes.data_as(C.c_void_p), recs.shape[0], out.ctypes.data_as(C.c_void_p))
        return out

    def observe(self, recs, agent, view, cropped=False):
        rb = (4 * (2 * view + 1) ** 2 + 12 + 31) & ~31 if cropped else 512
        out = np.zeros((recs.shape[0], rb), np.uint8)
        self.lib.radiosim_observe(recs.ctypes.data_as(C.c_void_p), recs.shape[0], agent, view, int(cropped),
                                  out.ctypes.data_as(C.c_void_p))
        return out


@pytest.fixture(scope="module")
def radiosim_so(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("radiosim") / "libradiosim.so")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-I", os.path.join(ROOT, "include"),
                          "-I", os.path.join(ROOT, "pomcpp_b200", "csrc"), "-o", so, os.path.join(HERE, "radiosim", "radiosim.cpp")],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return so


def _msgs(rng, n):
    """random message bytes, high bits included (the device ignores bits 6..7)"""
    return rng.integers(0, 256, (n, 4), dtype=np.uint8)


# ----------------------------------------------------------------------------------------------------------- CPU


def test_message_packing():
    """pack_messages / unpack_messages: [n, 4, 2] words <-> the byte encoding w0 | w1 << 3; bits 6..7 are ignored"""
    import pomcpp_b200 as pb
    w = np.random.default_rng(1).integers(0, 8, (50, 4, 2), dtype=np.uint8)
    m = pb.pack_messages(w)
    assert m.shape == (50, 4) and (m < 64).all() and (m == w[:, :, 0] + 8 * w[:, :, 1]).all()
    assert (pb.unpack_messages(m) == w).all()
    assert (pb.unpack_messages(m | 0xC0) == w).all()


def test_init_record_leaves_radio_zero(radiosim_so):
    """the device templates' generator (pomcore::init_record) clears the radio bytes: every episode starts silent"""
    sim = RadioSim(radiosim_so)
    out = np.full(3, 0xFF, np.uint8)
    for seed in (0x1337, 1, 99):
        sim.lib.radiosim_init_record_radio(seed, out.ctypes.data_as(C.c_void_p))
        assert (out == 0).all()


@pytest.mark.parametrize("kind,autoreset", [("random", True), ("harmless", True), ("stress", True), ("random", False),
                                            ("stress", False)])
def test_radio_latch_on_games(orc, radiosim_so, kind, autoreset):
    """games from InitState with auto-reset and max_ticks = 60 (or frozen at their end), random message bytes: status,
    rewards and messages == the restatement on every tick, every field every 25 ticks"""
    n, ticks, env0, max_ticks = 1024, 200, 7, 60
    nact = 5 if kind == "harmless" else 6
    rng = np.random.default_rng(31 + autoreset)
    S = _games(orc, n, stress=kind == "stress", seed=5)
    T = _games(orc, 48)
    R = RadioRestatement(orc, S, T, env0, max_ticks, autoreset)
    sim = RadioSim(radiosim_so, T, env0, max_ticks, autoreset)
    recs, bad = sim.h.pack(S)
    assert not bad.any()
    episodes = np.zeros(n, np.uint32)
    seen = {"dead_silent": 0, "reset": 0, "frozen": 0}
    for t in range(ticks):
        mv = orc.rng_moves(99 + t % 3, env0, n, t, nact)
        msgs = _msgs(rng, n)
        frozen = (R.status & (DONE | INVALID)) != 0
        end, want = R.tick(mv, msgs)
        st, rw = sim.tick(recs, episodes, mv, msgs)
        assert (st == end).all(), "status, tick %d env %d" % (t, np.nonzero(st != end)[0][0])
        assert (rw == want).all(), "rewards, tick %d" % t
        got = sim.messages(recs)
        assert (got == R.M).all(), "messages, tick %d env %d" % (t, np.nonzero((got != R.M).any(1))[0][0])
        if t % 25 == 24:
            assert orc.diff_batch(sim.h.unpack(recs)[0], R.S)[0] == -1, "tick %d" % t
        seen["dead_silent"] += int(((R.S["agents"]["dead"] != 0) & (R.M == 0) & ((msgs & 63) != 0)).sum())
        seen["reset"] += int((((end & (DONE | TRUNC | INVALID)) != 0) & ~frozen).sum())
        seen["frozen"] += int(frozen.sum())
    assert seen["reset"] > 0, seen
    if kind != "harmless":
        assert seen["dead_silent"] > 0, seen
    if not autoreset:
        assert seen["frozen"] > 0, seen


@pytest.mark.parametrize("autoreset", [False, True], ids=["frozen", "autoreset"])
def test_radio_latch_on_inconsistent_states(orc, radiosim_so, autoreset):
    """uploaded states no game reaches (tests/test_fuzz_states.py), a fifth uploaded done or invalid: messages == the
    restatement on the restated status and dead flags"""
    from test_fuzz_states import mutated_states
    from hostsim import HostSim
    S = mutated_states(orc, 611, 3000)
    rng = np.random.default_rng(4)
    n0 = S.shape[0]
    st0 = np.where(rng.random(n0) < 0.1, DONE | (1 << 2), np.where(rng.random(n0) < 0.1, INVALID, 0)).astype(np.uint8)
    recs, bad = HostSim().pack(S, st0)
    S, recs, st0 = S[bad == 0].copy(), recs[bad == 0].copy(), st0[bad == 0].copy()
    n = S.shape[0]
    assert n > 1500
    T = S[:16].copy()
    sim = RadioSim(radiosim_so, T, 0, 20, autoreset)
    R = RadioRestatement(orc, S, T, 0, 20, autoreset)
    R.status[:] = st0
    episodes = np.zeros(n, np.uint32)
    for t in range(16):
        mv = orc.rng_moves(77, 0, n, t, 6)
        msgs = _msgs(rng, n)
        end, _ = R.tick(mv, msgs)
        st, _ = sim.tick(recs, episodes, mv, msgs)
        invalid = (end & INVALID) != 0
        assert ((st & (DONE | INVALID)) == (end & (DONE | INVALID))).all() and (st[~invalid] == end[~invalid]).all(), "tick %d" % t
        got = sim.messages(recs)
        assert (got == R.M).all(), "messages, tick %d env %d" % (t, np.nonzero((got != R.M).any(1))[0][0])


def _case(orc, sim_so, killed=(), status0=0, max_ticks=0, autoreset=True, msgs=(0x3F, 0x01, 0x2A, 0x07), prep=None, ticks=1,
          m0=(0, 0, 0, 0)):
    """one team game from InitState with `killed` dead and last messages m0, IDLE moves, the same message bytes every
    tick: the messages after each tick from the host build of the kernel, checked against the restatement on the way"""
    S = _games(orc, 1)
    if killed:
        orc.kill(S, *killed)
    if prep:
        prep(orc, S)
    sim = RadioSim(sim_so, S.copy(), 0, max_ticks, autoreset)
    recs, bad = sim.h.pack(S, np.array([status0], np.uint8))
    assert not bad.any()
    v = sum(int(m) << (6 * a) for a, m in enumerate(m0))
    recs[0, 289:292] = [v & 0xFF, (v >> 8) & 0xFF, v >> 16]
    R = RadioRestatement(orc, S.copy(), S.copy(), 0, max_ticks, autoreset)
    R.status[:] = status0
    R.M[:] = sim.messages(recs)
    episodes = np.zeros(1, np.uint32)
    m = np.array([msgs], np.uint8)
    out = []
    for _ in range(ticks):
        R.tick(np.zeros((1, 4), np.uint8), m)
        sim.tick(recs, episodes, np.zeros((1, 4), np.uint8), m)
        got = sim.messages(recs)
        assert (got == R.M).all()
        out.append(got[0].tolist())
    return out


def _flame_on_agent1(orc, S):
    """agent 1 stands on a bomb that explodes in the next tick (its corner cell x = 10, y = 0): it dies in that tick"""
    orc.plant_bomb(S[0:1], 10, 0, 1, life=1)


@pytest.mark.parametrize("args,want", [
    (dict(), [[0x3F, 0x01, 0x2A, 0x07]]),                                                   # everyone sends
    (dict(killed=(1,), ticks=2), [[0x3F, 0, 0x2A, 0x07]] * 2),                             # a dead sender is silent
    (dict(prep=_flame_on_agent1, ticks=2), [[0x3F, 0x01, 0x2A, 0x07], [0x3F, 0, 0x2A, 0x07]]),  # dies this tick: sent
    (dict(status0=DONE | (1 << 2), ticks=2, m0=(9, 0, 5, 63)), [[9, 0, 5, 63]] * 2),       # frozen env: unchanged
    (dict(status0=INVALID, m0=(1, 2, 3, 4)), [[1, 2, 3, 4]]),                              # invalid env: unchanged
    (dict(killed=(0, 2), m0=(1, 2, 3, 4)), [[0, 0, 0, 0]]),                                # team 1 wins: the reset tick
    (dict(killed=(0, 2), autoreset=False, ticks=2), [[0, 0x01, 0, 0x07]] * 2),             # ... or frozen after it
    (dict(max_ticks=1), [[0, 0, 0, 0]]),                                                   # truncation resets too
    (dict(msgs=(0xFF, 0x40, 0x80 | 0x12, 0xC7)), [[0x3F, 0, 0x12, 0x07]]),                 # bits 6..7 ignored
], ids=["all-send", "dead-sender", "dies-this-tick", "frozen-done", "frozen-invalid", "reset-tick", "win-frozen",
        "truncation-reset", "high-bits"])
def test_radio_latch_cases(orc, radiosim_so, args, want):
    assert _case(orc, radiosim_so, **args) == want


@pytest.mark.parametrize("cropped", [False, True], ids=["full", "cropped"])
def test_radio_observation_layouts(orc, radiosim_so, cropped):
    """observe_planes<RADIO> / observe_cropped<RADIO> == the oracle's planes plus the teammate's two words, for every
    agent at views 0..5, on mid-game records whose radio bytes hold random messages"""
    from test_teams import _mid_game
    S = _mid_game(orc, 400, 8)
    sim = RadioSim(radiosim_so)
    recs, bad = sim.h.pack(S)
    S, recs = S[bad == 0].copy(), recs[bad == 0].copy()
    n = S.shape[0]
    rng = np.random.default_rng(12)
    M = rng.integers(0, 64, (n, 4), dtype=np.uint8)
    v = M[:, 0].astype(np.uint32) | (M[:, 1].astype(np.uint32) << 6) | (M[:, 2].astype(np.uint32) << 12) | (M[:, 3].astype(np.uint32) << 18)
    recs[:, 289], recs[:, 290], recs[:, 291] = v & 0xFF, (v >> 8) & 0xFF, v >> 16
    assert (sim.messages(recs) == M).all()
    nonzero = 0
    for view in range(6):
        for agent in range(4):
            want = radio_planes(orc, S, M, agent, view, cropped)
            got = sim.observe(recs, agent, view, cropped)
            assert (got == want).all(), "view %d agent %d env %d" % (view, agent, np.nonzero((got != want).any(1))[0][0])
            at = 4 * (2 * view + 1) ** 2 + 9 if cropped else 493
            nonzero += int((got[:, at] != 0).sum() + (got[:, at + 1] != 0).sum())
    assert nonzero > 0


# ----------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


def _to_dev(pb, dst, a):
    pb.lib().pom_device_copy(0, dst, a.ctypes.data_as(C.c_void_p), a.nbytes)


def _from_dev(pb, a, src):
    pb.lib().pom_device_copy(0, a.ctypes.data_as(C.c_void_p), src, a.nbytes)
    return a


def _ended(st):
    return (st & (DONE | TRUNC | INVALID)) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["autoreset", "no-autoreset", "continue-undefined", "mapped", "no-rewards"])
def test_step_radio_matches_restatement_and_twin(pb, orc, variant):
    """4099 envs (a partial last slice), max_ticks = 40: every tick the messages (radio_download), rewards and status bytes
    are the restatement's, computed from the twin non-radio team handle driven by step_rewards with the same moves; the
    full and cropped planes every 8 ticks; records, status bytes and counters bit-identical to the twin"""
    n, ticks = 4099, 120 if variant == "autoreset" else 60
    flags = {"no-autoreset": pb.STEP_COUNT,
             "continue-undefined": pb.STEP_AUTORESET | pb.STEP_COUNT | pb.STEP_CONTINUE_UNDEFINED}.get(variant, pb.STEP_AUTORESET | pb.STEP_COUNT)
    a = pb.Batch(n, n_templates=64, max_ticks=40, teams=True, radio=True)
    c = pb.Batch(n, n_templates=64, max_ticks=40, teams=True)
    assert a.radio() and a.teams() and not c.radio()
    rng = np.random.default_rng(17)
    owners = []
    if variant == "mapped":
        mv, o1 = pb.pinned_array((n, 4), np.uint8)
        ms, o2 = pb.pinned_array((n, 4), np.uint8)
        rw, o3 = pb.pinned_array((n, 4), np.int8)
        st, o4 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2, o3, o4]
        mv_a, ms_a, rw_a, st_a = mv, ms, rw, st
    else:
        mv, ms, rw, st = np.zeros((n, 4), np.uint8), np.zeros((n, 4), np.uint8), np.zeros((n, 4), np.int8), np.zeros(n, np.uint8)
        mv_a, ms_a, rw_a, st_a = a.alloc(4 * n), a.alloc(4 * n), a.alloc(4 * n), a.alloc(n)
    mv_c, rw_c, st_c = c.alloc(4 * n), c.alloc(4 * n), c.alloc(n)
    M = np.zeros((n, 4), np.uint8)
    assert (a.radio_download() == 0).all()
    counts = {"sent": 0, "silenced": 0, "reset": 0}
    S0, s0 = c.download()
    for t in range(ticks):
        mv[:] = rng.integers(0, 6, (n, 4), dtype=np.uint8)
        ms[:] = _msgs(rng, n)
        if variant != "mapped":
            _to_dev(pb, mv_a, mv)
            _to_dev(pb, ms_a, ms)
        _to_dev(pb, mv_c, mv)
        a.step_radio(mv_a, ms_a, None if variant == "no-rewards" else rw_a, st_a, flags)
        c.step_rewards(mv_c, rw_c, st_c, flags)
        a.sync(); c.sync()
        if variant != "mapped":
            if variant != "no-rewards":
                _from_dev(pb, rw, rw_a)
            _from_dev(pb, st, st_a)
        twin_st, twin_rw = _from_dev(pb, np.zeros(n, np.uint8), st_c), _from_dev(pb, np.zeros((n, 4), np.int8), rw_c)
        assert (st == twin_st).all(), "status, tick %d" % t
        if variant != "no-rewards":
            assert (rw == twin_rw).all(), "rewards, tick %d" % t
        S1, s1 = c.download()
        stepped = (s0 & (DONE | INVALID)) == 0
        alive = S0["agents"]["dead"] == 0
        M[stepped] = np.where(alive[stepped], ms[stepped] & 63, 0)
        if flags & pb.STEP_AUTORESET:
            M[stepped & _ended(twin_st)] = 0
            counts["reset"] += int((stepped & _ended(twin_st)).sum())
        want_rw = reward_definition(stepped, twin_st, S1["agents"]["dead"] != 0, True)
        assert (twin_rw == want_rw).all(), "rewards definition, tick %d" % t
        got = a.radio_download()
        assert (got == M).all(), "messages, tick %d env %d" % (t, np.nonzero((got != M).any(1))[0][0])
        counts["sent"] += int((M != 0).sum())
        counts["silenced"] += int((stepped[:, None] & ~alive & ((ms & 63) != 0)).sum())
        if t % 8 == 7:
            Sa, sa = a.download()
            assert Sa.tobytes() == S1.tobytes() and (sa == s1).all(), "records, tick %d" % t
            view, mask = t % 6, [15, 0b0101, 0b1010, 0b0110][(t // 8) % 4]
            agents = [x for x in range(4) if mask >> x & 1]
            full = a.observe_planes(mask, view)
            crop = a.observe_planes_cropped(mask, view)
            for k, ag in enumerate(agents):
                assert (full[k] == radio_planes(orc, Sa, M, ag, view)).all(), "full planes, tick %d agent %d" % (t, ag)
                assert (crop[k] == radio_planes(orc, Sa, M, ag, view, True)).all(), "cropped planes, tick %d agent %d" % (t, ag)
        S0, s0 = S1, s1
    assert (a.stats().as_array() == c.stats().as_array()).all(), (a.stats().as_dict(), c.stats().as_dict())
    assert counts["sent"] > 0 and counts["silenced"] > 0, counts
    if flags & pb.STEP_AUTORESET:
        assert counts["reset"] > 0, counts
    for o in owners:
        pb.pinned_free(o)
    if variant != "mapped":
        for p in (mv_a, ms_a, rw_a, st_a):
            a.free(p)
    for p in (mv_c, rw_c, st_c):
        c.free(p)
    a.close(); c.close()


def _other_entry_points(pb, a, n, rng, mv_dev, mv):
    """(name, call, ticks, resets, frozen) for every entry point besides step_radio that touches a radio handle's envs:
    `call()` runs it once; resets = whether it auto-resets envs that end; frozen = the status bits that keep an env from
    being stepped (the fused rollout kernel, which also runs step_seq, freezes a TRUNCATED env, which a frozen no-reset
    rollout leaves behind; the per-tick step steps it and resets it)"""
    AR = pb.STEP_AUTORESET | pb.STEP_COUNT
    K, R = DONE | INVALID, DONE | INVALID | TRUNC
    joint, o1 = pb.pinned_array((n,), np.uint16)
    done_bits, o2 = pb.pinned_array(((n + 31) // 32,), np.uint32)
    status, o3 = pb.pinned_array((n,), np.uint8)
    seq = a.alloc(4 * n * 5)
    for k in range(5):
        a.generate_moves(seq.value + 4 * n * k, 3, 50 + k, 6)
    obs = a.alloc(2 * int(pb.lib().pom_batch_obs_stride(a.h)) * pb.OBS_BYTES)
    rw, st = a.alloc(4 * n), a.alloc(n)

    def compact():
        joint[:] = pb.joint_of_moves(mv)
        a.step_compact(joint, done_bits=done_bits, flags=AR)
    calls = [
        ("step", lambda: a.step(mv_dev, AR), 1, True, K),
        ("step-no-reset", lambda: a.step(mv_dev, pb.STEP_COUNT), 1, False, K),
        ("step_host", lambda: a.step_host(mv, status, AR), 1, True, K),
        ("step_compact", compact, 1, True, K),
        ("step_observe", lambda: a.step_observe(mv_dev, obs, 0b0101, 4, AR), 1, True, K),
        ("step_rewards", lambda: a.step_rewards(mv_dev, rw, st, AR), 1, True, K),
        ("step_seq", lambda: a.step_seq(seq, 5, 0), 5, True, R),
        ("step_seq-no-reset", lambda: a.step_seq(seq, 5, pb.ROLL_NO_RESET), 5, False, R),
        ("rollout", lambda: a.rollout(1, 7, 0, 0), 1, True, R),
        ("rollout-no-reset", lambda: a.rollout(6, 7, 0, pb.ROLL_NO_RESET), 6, False, R),
        ("rollout-simple", lambda: a.rollout(1, 9, 0, pb.ROLL_SIMPLE(0b0111)), 1, True, R),
        ("rollout-simple-no-reset", lambda: a.rollout(4, 9, 0, pb.ROLL_SIMPLE(0b1111) | pb.ROLL_NO_RESET), 4, False, R),
        ("policy_moves", lambda: a.policy_moves(mv_dev, 5, 0, 15), 0, False, K),
    ]
    return calls, (o1, o2, o3), (seq, obs, rw, st)


@pytest.mark.gpu
def test_other_entry_points_keep_or_clear_messages(pb):
    """on a radio handle of 4099 envs with random last messages: every other stepping or acting call leaves the messages
    of envs it does not re-initialise as they were and clears those it auto-resets; the game is not touched by the
    radio (states equal to a non-radio twin that gets the same calls); clone copies, expand_step children inherit, upload
    and reset clear"""
    n = 4099
    a = pb.Batch(n, n_templates=64, max_ticks=40, teams=True, radio=True)
    c = pb.Batch(n, n_templates=64, max_ticks=40, teams=True)
    rng = np.random.default_rng(23)
    a.rollout(100, 3, 0, 0)                                    # every phase of a game, some envs near their time limit
    c.rollout(100, 3, 0, 0)
    mv = np.ascontiguousarray(rng.integers(0, 6, (n, 4), dtype=np.uint8))
    mv_dev = a.alloc(4 * n)
    _to_dev(pb, mv_dev, mv)
    calls, owners, bufs = _other_entry_points(pb, a, n, rng, mv_dev, mv)
    twin, twin_owners, twin_bufs = _other_entry_points(pb, c, n, rng, mv_dev, mv)
    twin_calls = dict((k, f) for k, f, _, _, _ in twin)
    resets = 0
    for name, call, ticks, autoreset, frozen in calls:
        M = rng.integers(0, 64, (n, 4), dtype=np.uint8)
        a.radio_upload(M)
        S0, s0 = a.download()
        call()
        twin_calls[name]()
        a.sync(); c.sync()
        S1, s1 = a.download()
        Sc, sc = c.download()
        assert S1.tobytes() == Sc.tobytes() and (s1 == sc).all(), name
        running = (s0 & frozen) == 0
        # an env re-initialised by an auto-reset holds a template: its timeStep is below what `ticks` ticks give
        reset = running & (S1["timeStep"] < S0["timeStep"] + ticks) if autoreset else np.zeros(n, bool)
        want = np.where(reset[:, None], 0, M)
        got = a.radio_download()
        assert (got == want).all(), "%s: env %d" % (name, np.nonzero((got != want).any(1))[0][0])
        resets += int(reset.sum())
    assert resets > 0
    # clone copies, expand_step children inherit their root's messages
    M = rng.integers(0, 64, (n, 4), dtype=np.uint8)
    a.radio_upload(M)
    d = pb.Batch(360, n_templates=8, teams=True, radio=True)
    idx = rng.integers(0, n, 200).astype(np.uint32)
    d.clone_from(a, idx, first_dst=100)
    d.sync()
    got = d.radio_download()
    assert (got[100:300] == M[idx]).all() and (got[:100] == 0).all() and (got[300:] == 0).all()
    roots = rng.integers(0, n, 10).astype(np.uint32)
    d.expand_step_from(a, roots, fanout=36)
    d.sync()
    assert (d.radio_download() == np.repeat(M[roots], 36, axis=0)).all()
    # upload and reset re-initialise
    S, st = a.download(first=0, count=500)
    a.upload(S, st, first=1000)
    got = a.radio_download()
    assert (got[1000:1500] == 0).all() and (got[:1000] == M[:1000]).all() and (got[1500:] == M[1500:]).all()
    a.reset()
    assert (a.radio_download() == 0).all()
    for o in owners + twin_owners:
        pb.pinned_free(o)
    for p in bufs + (mv_dev,):
        a.free(p)
    for p in twin_bufs:
        c.free(p)
    d.close(); a.close(); c.close()


@pytest.mark.gpu
def test_radio_planes_are_never_fused(pb, monkeypatch):
    """with POM_OBS_FUSED=1 a radio handle's step_observe and step_compact still queue the observation kernel: the planes
    are those of observe_planes (with the messages) after the same tick"""
    n = 4099
    monkeypatch.setenv("POM_OBS_FUSED", "1")
    a = pb.Batch(n, n_templates=64, max_ticks=40, teams=True, radio=True)
    monkeypatch.delenv("POM_OBS_FUSED")
    rng = np.random.default_rng(5)
    a.rollout(30, 3, 0, 0)
    a.radio_upload(rng.integers(0, 64, (n, 4), dtype=np.uint8))
    mv_dev = a.alloc(4 * n)
    stride = int(pb.lib().pom_batch_obs_stride(a.h))
    obs = a.alloc(2 * stride * pb.OBS_BYTES)
    a.generate_moves(mv_dev, 1, 0, 6)
    a.step_observe(mv_dev, obs, 0b0110, 3, pb.STEP_AUTORESET)
    a.sync()
    got = _from_dev(pb, np.zeros((2, stride, pb.OBS_BYTES), np.uint8), obs)[:, :n]
    want = a.observe_planes(0b0110, 3)
    assert (got == want).all() and (want[:, :, 493:495] != 0).any()
    joint, o = pb.pinned_array((n,), np.uint16)
    joint[:] = rng.integers(0, 1296, n)
    a.step_compact(joint, flags=pb.STEP_AUTORESET, obs_dev=obs, obs_agent_mask=0b1001, obs_view=4)
    a.sync()
    got = _from_dev(pb, np.zeros((2, stride, pb.OBS_BYTES), np.uint8), obs)[:, :n]
    assert (got == a.observe_planes(0b1001, 4)).all()
    pb.pinned_free(o)
    a.free(mv_dev); a.free(obs)
    a.close()


@pytest.mark.gpu
def test_radio_refusals(pb, monkeypatch):
    """POM_E_ARG, with nothing stepped: a radio handle without the team game, step_radio on a handle without the radio,
    RAW, OVERLAP and unknown flags, null moves or messages, pageable buffers, misaligned messages or rewards, a handle
    made with POM_STEP_KERNEL=tile; radio_download / upload on a handle without the radio; clone and expand_step between
    a radio and a non-radio handle"""
    L = pb.lib()
    n = 300
    with pytest.raises(pb.PomError):
        pb.Batch(n, n_templates=8, radio=True)
    b = pb.Batch(n, n_templates=8, teams=True, radio=True)
    t = pb.Batch(n, n_templates=8, teams=True)
    assert L.pom_batch_radio(b.h) == 1 and L.pom_batch_radio(t.h) == 0 and L.pom_batch_radio(None) == -1
    mv, ms, rw, st = b.alloc(4 * n), b.alloc(4 * n), b.alloc(4 * n), b.alloc(n)
    b.generate_moves(mv, 1, 0, 6)
    b.generate_moves(ms, 2, 0, 6)
    S0, s0 = b.download()
    page = np.zeros(4 * n, np.uint8)
    pp = page.ctypes.data_as(C.c_void_p)
    for f in (pb.STEP_RAW, pb.STEP_OVERLAP, pb.STEP_AUTORESET | pb.STEP_RAW, 0x40000000, 0x20):
        assert L.pom_batch_step_radio(b.h, mv, ms, f, rw, st) == -1, f
    assert L.pom_batch_step_radio(t.h, mv, ms, 0, rw, st) == -1 and b"POM_INIT_RADIO" in L.pom_last_error()
    assert L.pom_batch_step_radio(b.h, None, ms, 0, rw, st) == -1
    assert L.pom_batch_step_radio(b.h, mv, None, 0, rw, st) == -1
    assert L.pom_batch_step_radio(b.h, pp, ms, 0, rw, st) == -1
    assert L.pom_batch_step_radio(b.h, mv, pp, 0, rw, st) == -1
    assert L.pom_batch_step_radio(b.h, mv, ms, 0, pp, st) == -1
    assert L.pom_batch_step_radio(b.h, mv, ms, 0, rw, pp) == -1
    assert L.pom_batch_step_radio(b.h, mv, C.c_void_p(ms.value + 1), 0, rw, st) == -1 and b"aligned" in L.pom_last_error()
    assert L.pom_batch_step_radio(b.h, mv, ms, 0, C.c_void_p(rw.value + 2), st) == -1 and b"aligned" in L.pom_last_error()
    assert L.pom_batch_step_radio(None, mv, ms, 0, rw, st) == -1
    S1, s1 = b.download()
    assert S1.tobytes() == S0.tobytes() and (s1 == s0).all() and b.stats().env_steps == 0 and (b.radio_download() == 0).all()
    assert L.pom_batch_step_radio(b.h, mv, ms, pb.STEP_COUNT, None, None) == 0
    b.sync()
    assert b.stats().env_steps == n and (b.radio_download() != 0).any()
    buf = np.zeros((n, 4), np.uint8)
    bp = buf.ctypes.data_as(C.c_void_p)
    assert L.pom_batch_radio_download(t.h, 0, n, bp) == -1 and L.pom_batch_radio_upload(t.h, 0, n, bp) == -1
    assert L.pom_batch_radio_download(b.h, 0, n, None) == -1 and L.pom_batch_radio_upload(b.h, 0, n, None) == -1
    assert L.pom_batch_radio_download(b.h, 1, n, bp) == -4 and L.pom_batch_radio_upload(b.h, 1, n, bp) == -4
    idx = np.zeros(4, np.uint32)
    assert L.pom_batch_clone(t.h, 0, b.h, idx.ctypes.data_as(C.c_void_p), 4) == -1 and b"radio" in L.pom_last_error()
    assert L.pom_batch_clone(b.h, 0, t.h, idx.ctypes.data_as(C.c_void_p), 4) == -1
    assert L.pom_batch_expand_step(t.h, b.h, idx.ctypes.data_as(C.c_void_p), 1, 36, 0) == -1 and b"radio" in L.pom_last_error()
    assert L.pom_batch_expand_step(b.h, t.h, idx.ctypes.data_as(C.c_void_p), 1, 36, 0) == -1
    monkeypatch.setenv("POM_STEP_KERNEL", "tile")
    k = pb.Batch(n, n_templates=8, teams=True, radio=True)
    monkeypatch.delenv("POM_STEP_KERNEL")
    assert L.pom_batch_step_radio(k.h, mv, ms, 0, rw, st) == -1 and b"POM_STEP_KERNEL" in L.pom_last_error()
    for p in (mv, ms, rw, st):
        b.free(p)
    b.close(); t.close(); k.close()


BATCH_ENV_CPP = r"""
#include <cstdio>
#include <cstring>
#include <vector>
#include "pom_bboard.hpp"
using namespace bboard;
int main()
{
    const size_t n = 4096;
    BatchEnvironment env(n, 0, 0, 64, 0x1337, 0, true, true), plain(n, 0, 0, 64, 0x1337, 0, true);
    if(!env.HasRadio() || plain.HasRadio()) return 1;
    std::vector<Move> mv(4 * n);
    std::vector<uint8_t> msg(4 * n);
    std::vector<int8_t> rw(4 * n), rw_plain(4 * n);
    long heard = 0;
    for(uint32_t t = 0; t < 200; t++)
    {
        for(size_t e = 0; e < n; e++)
        {
            const uint32_t m = pom_rng_moves(5, e, t, 6), w = pom_rng_moves(6, e, t, 64);
            for(int a = 0; a < 4; a++) { mv[4 * e + a] = Move((m >> (8 * a)) & 0xFF); msg[4 * e + a] = uint8_t((w >> (8 * a)) & 0xFF); }
        }
        const std::vector<State> before = env.States();
        const std::vector<uint8_t> st0 = env.Status();
        const size_t running = t % 2 ? env.StepRadio(mv.data(), msg.data(), rw.data()) : env.StepRadio(mv.data(), msg.data());
        if(running != plain.Step(mv.data(), rw_plain.data())) return 2;
        if(t % 2 && std::memcmp(rw.data(), rw_plain.data(), 4 * n) != 0) return 3;
        for(size_t i = 0; i < n; i += 97)
        {
            const bool stepped = !(st0[i] & (POM_STATUS_DONE | POM_STATUS_INVALID));
            const bool ended = env.Status()[i] & (POM_STATUS_DONE | POM_STATUS_TRUNCATED | POM_STATUS_INVALID);
            if(!stepped || ended) continue;
            for(int a = 0; a < 4; a++)
            {
                const int m = before[i].agents[a].dead ? 0 : msg[4 * i + a];
                const std::pair<int, int> w = env.GetMessage(i, a);
                if(w.first != (m & 7) || w.second != (m >> 3)) return 4;
                heard += m != 0;
            }
        }
    }
    const std::vector<State> a = env.States(), b = plain.States();
    for(size_t i = 0; i < n; i++) if(std::memcmp(&a[i], &b[i], sizeof(State)) != 0) return 5;
    std::printf("%ld\n", heard);
    return 0;
}
"""


@pytest.mark.gpu
def test_batch_environment_step_radio(pb, tmp_path):
    """bboard::BatchEnvironment::StepRadio == Step(moves, rewards) on a non-radio team game for states, rewards and the
    running count; GetMessage reads back what a live agent of a stepped game sent"""
    src, exe = tmp_path / "radio_env.cpp", tmp_path / "radio_env"
    src.write_text(BATCH_ENV_CPP)
    lib = os.path.join(ROOT, "pomcpp_b200")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                          os.path.join(lib, "host", "libpom_host.a"), "-L" + lib, "-lpom_b200", "-Wl,-rpath," + lib],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert int(run.stdout) > 0
