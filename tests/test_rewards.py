"""Per-agent rewards of the per-tick step (pom_batch_step_rewards).  The reference has no reward, so this file holds the
definition in two forms and pins the device code to it:
  reward_definition   the status-byte form of include/pom_batch.h: from `stepped`, the end-of-tick status byte before
                      any auto-reset and the agents' dead flags.  It alone governs inconsistent uploaded states, where
                      aliveAgents and the dead flags can disagree.
  RewardRestatement   Pommerman's alive-list form (the reward function of the Pommerman Python environment) on the
                      restated state: count the live agents, then apply the free-for-all or team cases.  On every state a
                      game reaches the two forms agree.
  CPU  tests/rewardsim (pomcore::tick_rewards over records stepped by the device code built for the host, with the
       per-tick kernel's truncation and auto-reset) == both forms, on random, harmless, stress and inconsistent states,
       and on explicit cases.
  GPU  pom_batch_step_rewards on free-for-all and team handles == the definition on every tick, with states, status bytes
       and counters bit-identical to a twin handle driven by pom_batch_step_host with the same moves; the refusals;
       bboard::BatchEnvironment::Step(moves, rewards)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_teams import TeamRestatement, _games

DONE, DRAW, INVALID, TRUNC = 0x01, 0x02, 0x10, 0x20
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TEAM_OF = np.arange(4) & 1


def reward_definition(stepped, st, dead, teams):
    """[n, 4] int8 rewards from the status-byte form: first matching case of
         not stepped | st & INVALID      -> 0
         DONE, not DRAW, winner w        -> +1 for w (team game: team w), -1 for the others
         DONE | DRAW, TRUNCATED          -> -1
         running                         -> free-for-all: -1 if dead else 0; team game: 0"""
    st = np.asarray(st).astype(np.int64)
    w = (st >> 2) & 3
    winners = (TEAM_OF[None, :] == (w[:, None] & 1)) if teams else (np.arange(4)[None, :] == w[:, None])
    won = (st & (DONE | DRAW)) == DONE
    over = (st & (DONE | TRUNC)) != 0
    running = np.zeros((st.shape[0], 4), np.int64) if teams else -np.asarray(dead, bool).astype(np.int64)
    r = np.where(won[:, None], np.where(winners, 1, -1), np.where(over[:, None], -1, running))
    r[~np.asarray(stepped, bool) | ((st & INVALID) != 0)] = 0
    return r.astype(np.int8)


class RewardRestatement:
    """Pommerman's reward function on the restated state after the tick (before any reset), alive-list form:
      free-for-all  one agent alive: +1 for it, -1 for the others; else time up (timeStep >= max_ticks) or nobody alive:
                    -1 for everyone; else 0 for the live agents and -1 for the dead ones
      team game     only agents of team 0 (of 0, 2) alive: +1, -1, +1, -1; only team 1: -1, +1, -1, +1; else time up or
                    nobody alive: -1 for everyone; else 0
    plus this project's two cases: an env that was not stepped, or whose episode was aborted (INVALID), gets 0.
    max_ticks = 0: no time limit (the per-tick kernel truncates only when it auto-resets)."""

    def __init__(self, teams, max_ticks=0):
        self.teams, self.max_ticks = teams, max_ticks

    def rewards(self, S, stepped, invalid):
        alive = S["agents"]["dead"] == 0
        k = alive.sum(1)
        up = ((S["timeStep"] >= self.max_ticks) if self.max_ticks else np.zeros(S.shape[0], bool)) | (k == 0)
        if self.teams:
            t0, t1 = alive[:, 0] | alive[:, 2], alive[:, 1] | alive[:, 3]
            r = np.where((t0 & ~t1)[:, None], [1, -1, 1, -1],
                         np.where((t1 & ~t0)[:, None], [-1, 1, -1, 1], np.where(up[:, None], -1, 0)))
        else:
            a = alive.astype(np.int64)
            r = np.where((k == 1)[:, None], 2 * a - 1, np.where(up[:, None], -1, a - 1))
        r[~stepped | invalid] = 0
        return r.astype(np.int8)


class RewardRun:
    """the restatement replaying pom_batch_step_rewards: Environment::Step (free-for-all or TeamRestatement), truncation
    at max_ticks, reset to template[(env_offset + e + episode) % n_templates], all when auto-resetting.  tick() returns
    the status bytes before the reset and the rewards of both forms of the definition."""

    def __init__(self, orc, S, T, teams, env0=0, max_ticks=0, autoreset=True):
        self.game = TeamRestatement(orc) if teams else orc
        self.S, self.T, self.teams, self.env0, self.autoreset = S, T, teams, env0, autoreset
        self.max_ticks = max_ticks if autoreset else 0
        self.status = np.zeros(S.shape[0], np.uint8)
        self.episode = np.zeros(S.shape[0], np.int64)

    def tick(self, mv):
        S, st = self.S, self.status
        stepped = (st & (DONE | INVALID)) == 0
        self.game.env_step_batch(S, st, np.ascontiguousarray(mv))
        if self.max_ticks:
            st[stepped & ((st & DONE) == 0) & (S["timeStep"] >= self.max_ticks)] |= TRUNC
        end = st.copy()
        want = reward_definition(stepped, end, S["agents"]["dead"] != 0, self.teams)
        alive_form = RewardRestatement(self.teams, self.max_ticks).rewards(S, stepped, (end & INVALID) != 0)
        if self.autoreset:
            for e in np.nonzero(stepped & ((end & (DONE | INVALID | TRUNC)) != 0))[0]:
                self.episode[e] += 1
                S[e] = self.T[(self.env0 + e + self.episode[e]) % self.T.shape[0]]
                st[e] = 0
        return end, want, alive_form


class RewardSim:
    """tests/rewardsim: one tick of pom_batch_step_rewards on packed records (records packed by tests/hostsim)"""

    def __init__(self, so, teams, templates=None, env0=0, max_ticks=0, autoreset=True):
        from hostsim import HostSim
        self.h = HostSim()
        L = self.lib = C.CDLL(so)
        vp = C.c_void_p
        L.rewardsim_tick.argtypes = [vp, C.c_long, vp, C.c_int, C.c_int, C.c_uint32, vp, C.c_long, C.c_uint64, vp, vp, vp]
        self.teams, self.env0, self.max_ticks, self.autoreset = teams, env0, max_ticks, autoreset
        self.tmpl = self.h.pack(templates)[0] if templates is not None else np.zeros((1, 292), np.uint8)

    def tick(self, recs, episodes, mv):
        n = recs.shape[0]
        st, rw = np.zeros(n, np.uint8), np.zeros((n, 4), np.int8)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.rewardsim_tick(p(recs), n, p(np.ascontiguousarray(mv)), int(self.teams), int(self.autoreset),
                                self.max_ticks, p(self.tmpl), self.tmpl.shape[0], self.env0, p(episodes), p(st), p(rw))
        return st, rw


@pytest.fixture(scope="module")
def rewardsim_so(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("rewardsim") / "librewardsim.so")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-I", os.path.join(ROOT, "include"),
                          "-I", os.path.join(ROOT, "pomcpp_b200", "csrc"), "-o", so, os.path.join(HERE, "rewardsim", "rewardsim.cpp")],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return so


# ----------------------------------------------------------------------------------------------------------- CPU


def test_definition_tables():
    """the status-byte form on hand-picked bytes, both modes"""
    dead = np.array([[0, 1, 0, 1]] * 9, bool)
    st = np.array([0, DONE | (2 << 2), DONE | (1 << 2), DONE | DRAW, TRUNC, INVALID | DONE | (1 << 2), INVALID, 0, DRAW], np.uint8)
    stepped = np.array([1, 1, 1, 1, 1, 1, 1, 0, 1], bool)
    ffa = reward_definition(stepped, st, dead, False)
    team = reward_definition(stepped, st, dead, True)
    assert ffa.tolist() == [[0, -1, 0, -1], [-1, -1, 1, -1], [-1, 1, -1, -1], [-1] * 4, [-1] * 4, [0] * 4, [0] * 4, [0] * 4,
                            [0, -1, 0, -1]]
    assert team.tolist() == [[0] * 4, [1, -1, 1, -1], [-1, 1, -1, 1], [-1] * 4, [-1] * 4, [0] * 4, [0] * 4, [0] * 4, [0] * 4]


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("kind,autoreset", [("random", True), ("harmless", True), ("stress", True), ("random", False)])
def test_tick_rewards_on_games(orc, rewardsim_so, teams, kind, autoreset):
    """games from InitState with auto-reset and max_ticks = 60 (or frozen at their end): status bytes, rewards == both
    forms of the definition on every tick, every field every 25 ticks"""
    n, ticks, env0, max_ticks = 1024, 200, 7, 60
    nact = 5 if kind == "harmless" else 6
    S = _games(orc, n, stress=kind == "stress", seed=5)
    T = _games(orc, 48)
    R = RewardRun(orc, S, T, teams, env0, max_ticks, autoreset)
    sim = RewardSim(rewardsim_so, teams, T, env0, max_ticks, autoreset)
    recs, bad = sim.h.pack(S)
    assert not bad.any()
    episodes = np.zeros(n, np.uint32)
    seen = {"win": 0, "lost_all": 0, "dead_running": 0, "trunc": 0}
    for t in range(ticks):
        mv = orc.rng_moves(99 + t % 3, env0, n, t, nact)
        end, want, alive_form = R.tick(mv)
        st, rw = sim.tick(recs, episodes, mv)
        assert (st == end).all(), "status, tick %d env %d" % (t, np.nonzero(st != end)[0][0])
        assert (want == alive_form).all(), "the two forms disagree, tick %d env %d" % (t, np.nonzero((want != alive_form).any(1))[0][0])
        assert (rw == want).all(), "rewards, tick %d env %d" % (t, np.nonzero((rw != want).any(1))[0][0])
        if t % 25 == 24:
            assert orc.diff_batch(sim.h.unpack(recs)[0], R.S)[0] == -1, "tick %d" % t
            assert (episodes == R.episode).all()
        seen["win"] += int((rw == 1).any(1).sum())
        seen["lost_all"] += int((rw == -1).all(1).sum())
        seen["dead_running"] += int(((rw == -1).any(1) & (rw == 0).any(1)).sum())
        seen["trunc"] += int(((end & TRUNC) != 0).sum())
    if kind != "harmless":
        assert seen["win"] > 0 and seen["lost_all"] > 0, seen
    if autoreset:
        assert seen["trunc"] > 0, seen
    assert (seen["dead_running"] > 0) == (not teams and kind != "harmless"), seen


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("autoreset", [False, True], ids=["frozen", "autoreset"])
def test_tick_rewards_on_inconsistent_states(orc, rewardsim_so, teams, autoreset):
    """uploaded states no game reaches (tests/test_fuzz_states.py), aliveAgents out of step with the dead flags in a third
    of them: rewards == the status-byte form (which alone governs here) on the restated status and dead flags"""
    from test_fuzz_states import mutated_states
    S = mutated_states(orc, 601 + teams, 3000)
    rng = np.random.default_rng(3)
    off = rng.random(S.shape[0]) < 0.33
    S["aliveAgents"][off] = rng.integers(0, 5, int(off.sum()))
    from hostsim import HostSim
    recs, bad = HostSim().pack(S, np.zeros(S.shape[0], np.uint8))
    S, recs = S[bad == 0].copy(), recs[bad == 0].copy()
    n = S.shape[0]
    assert n > 1500
    T = S[:16].copy()
    sim = RewardSim(rewardsim_so, teams, T, 0, 20, autoreset)
    R = RewardRun(orc, S, T, teams, 0, 20, autoreset)
    episodes = np.zeros(n, np.uint32)
    disagree = 0
    for t in range(16):
        mv = orc.rng_moves(77, 0, n, t, 6)
        end, want, alive_form = R.tick(mv)
        st, rw = sim.tick(recs, episodes, mv)
        invalid = (end & INVALID) != 0
        assert ((st & (DONE | INVALID)) == (end & (DONE | INVALID))).all() and (st[~invalid] == end[~invalid]).all(), "tick %d" % t
        assert (rw == want).all(), "tick %d env %d" % (t, np.nonzero((rw != want).any(1))[0][0])
        disagree += int((want != alive_form).any(1).sum())
    if not teams:
        assert disagree > 0                                  # the counter decides a free-for-all game, not the flags


def _case(orc, sim_so, teams, killed=(), status0=0, time=None, max_ticks=0, autoreset=True, ticks=1):
    """one game from InitState with `killed` dead, IDLE moves: (rewards, status) of each tick from the host build of the
    kernel, checked against the status-byte form on the way"""
    S = _games(orc, 1)
    if killed:
        orc.kill(S, *killed)
    if time is not None:
        S["timeStep"][0] = time
    sim = RewardSim(sim_so, teams, S.copy(), 0, max_ticks, autoreset)
    recs, bad = sim.h.pack(S, np.array([status0], np.uint8))
    assert not bad.any()
    episodes = np.zeros(1, np.uint32)
    out, prev = [], status0
    for _ in range(ticks):
        st, rw = sim.tick(recs, episodes, np.zeros((1, 4), np.uint8))
        G, now = sim.h.unpack(recs)
        # the record after a reset holds the template's dead flags: the definition reads them only while the game runs
        assert (rw == reward_definition(np.array([(prev & (DONE | INVALID)) == 0]), st, G["agents"]["dead"] != 0, teams)).all()
        out.append((rw[0].tolist(), int(st[0])))
        prev = int(now[0])
    return out


FFA_WIN, TEAM0_WIN = [1, -1, -1, -1], [1, -1, 1, -1]


@pytest.mark.parametrize("teams,args,want", [
    (False, dict(killed=(1, 2, 3)), [(FFA_WIN, DONE)]),
    (False, dict(killed=(0, 1, 2, 3)), [([-1] * 4, DONE | DRAW)]),
    (False, dict(killed=(2, 3), max_ticks=1), [([-1] * 4, TRUNC)]),                       # truncation with two alive
    (False, dict(killed=(1, 2, 3), max_ticks=1), [(FFA_WIN, DONE)]),                      # a win on the last tick is a win
    (False, dict(killed=(1,), ticks=4), [([0, -1, 0, 0], 0)] * 4),                        # a dead agent in a running game
    (False, dict(killed=(1, 2, 3), autoreset=False, ticks=3), [(FFA_WIN, DONE), ([0] * 4, DONE), ([0] * 4, DONE)]),
    (False, dict(killed=(1,), time=65535), [([0] * 4, INVALID)]),                         # the env becomes INVALID
    (False, dict(killed=(1, 2, 3), status0=DONE, ticks=2), [([0] * 4, DONE)] * 2),        # frozen env
    (True, dict(killed=(2,), ticks=4), [([0] * 4, 0)] * 4),                               # a dead teammate, game running
    (True, dict(killed=(0, 1, 3)), [(TEAM0_WIN, DONE)]),                                  # a team win by one survivor
    (True, dict(killed=(0, 2)), [([-1, 1, -1, 1], DONE | (1 << 2))]),
    (True, dict(killed=(0, 1, 2, 3)), [([-1] * 4, DONE | DRAW)]),
    (True, dict(killed=(2,), max_ticks=1), [([-1] * 4, TRUNC)]),
    (True, dict(status0=INVALID, ticks=2), [([0] * 4, INVALID)] * 2),                     # frozen env
], ids=["ffa-win", "ffa-draw", "ffa-truncated", "ffa-win-last-tick", "ffa-dead-running", "ffa-frozen-after-win",
        "ffa-invalid", "ffa-frozen-done", "team-dead-teammate", "team-win-one-survivor", "team1-win", "team-draw",
        "team-truncated", "team-frozen-invalid"])
def test_tick_rewards_cases(orc, rewardsim_so, teams, args, want):
    assert _case(orc, rewardsim_so, teams, **args) == want


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


def _drive(pb, a, c, teams, ticks, flags, seed, simple=False, mapped=False):
    """`ticks` ticks of a.step_rewards against c.step_host with the same moves (random, or SimpleAgents for agents 0..2
    through pom_batch_policy_moves on a): every tick the status bytes are equal and the rewards are the definition of the
    twin's status bytes and dead flags (after the reset: the definition reads them only while the game runs); every 20
    ticks and at the end the two handles' records, status bytes and counters are bit-identical.  Returns reward counts."""
    n = a.n
    rng = np.random.default_rng(seed)
    owners = []
    if mapped:
        mv, o1 = pb.pinned_array((n, 4), np.uint8)
        rw, o2 = pb.pinned_array((n, 4), np.int8)
        st, o3 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2, o3]
        mv_arg, rw_arg, st_arg = mv, rw, st
    else:
        mv, rw, st = np.zeros((n, 4), np.uint8), np.zeros((n, 4), np.int8), np.zeros(n, np.uint8)
        mv_arg, rw_arg, st_arg = a.alloc(4 * n), a.alloc(4 * n), a.alloc(n)
    twin = np.zeros(n, np.uint8)
    prev = c.status()
    counts = np.zeros(3, np.int64)
    for t in range(ticks):
        mv[:] = rng.integers(0, 6, (n, 4), dtype=np.uint8)
        if simple and mapped:
            a.policy_moves_host(mv, seed, t, 0b0111)
        elif simple:
            _to_dev(pb, mv_arg, mv)
            a.policy_moves(mv_arg, seed, t, 0b0111)
            a.sync()
            _from_dev(pb, mv, mv_arg)
        elif not mapped:
            _to_dev(pb, mv_arg, mv)
        a.step_rewards(mv_arg, rw_arg, st_arg if t % 4 else None, flags)
        c.step_host(mv, twin, flags)
        a.sync()
        if not mapped:
            _from_dev(pb, rw, rw_arg)
            if t % 4:
                _from_dev(pb, st, st_arg)
        S, cur = c.download()
        if t % 4:
            assert (st == twin).all(), "status, tick %d env %d" % (t, np.nonzero(st != twin)[0][0])
        want = reward_definition((prev & (DONE | INVALID)) == 0, twin, S["agents"]["dead"] != 0, teams)
        assert (rw == want).all(), "rewards, tick %d env %d: %s != %s" % (t, np.nonzero((rw != want).any(1))[0][0],
                                                                       rw[(rw != want).any(1)][0], want[(rw != want).any(1)][0])
        counts += [int((rw == 1).sum()), int((rw == -1).sum()), int((rw == 0).all(1).sum())]
        prev = cur
        if t % 20 == 19 or t == ticks - 1:
            Sa, sa = a.download()
            assert Sa.tobytes() == S.tobytes() and (sa == cur).all(), "records, tick %d" % t
    assert (a.stats().as_array() == c.stats().as_array()).all(), (a.stats().as_dict(), c.stats().as_dict())
    for o in owners:
        pb.pinned_free(o)
    if not mapped:
        for p in (mv_arg, rw_arg, st_arg):
            a.free(p)
    return counts


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("simple", [False, True], ids=["random", "simple-agents"])
def test_step_rewards_matches_definition_and_twin(pb, teams, simple):
    """4099 envs (a partial last slice), max_ticks = 40, auto-reset, 200 ticks"""
    n = 4099
    a = pb.Batch(n, n_templates=64, max_ticks=40, teams=teams)
    c = pb.Batch(n, n_templates=64, max_ticks=40, teams=teams)
    counts = _drive(pb, a, c, teams, 200, pb.STEP_AUTORESET | pb.STEP_COUNT, 11 + simple, simple=simple)
    s = c.stats()
    assert counts[0] > 0 and counts[1] > 0 and s.truncated > 0 and s.episodes > 0, (counts, s.as_dict())
    a.close(); c.close()


def _uploaded(pb, orc, n, teams, seed):
    """inconsistent states (aliveAgents off in a third) with a tenth uploaded done, a tenth invalid"""
    from hostsim import HostSim
    from test_fuzz_states import mutated_states
    S = mutated_states(orc, seed, n + 3000)
    rng = np.random.default_rng(seed)
    off = rng.random(S.shape[0]) < 0.33
    S["aliveAgents"][off] = rng.integers(0, 5, int(off.sum()))
    bad = HostSim().pack(S)[1]
    S = np.ascontiguousarray(S[bad == 0][:n])
    assert S.shape[0] == n
    u = rng.random(n)
    st = np.where(u < 0.1, DONE | (1 << 2), np.where(u < 0.2, INVALID, np.where(u < 0.25, DONE | DRAW, 0))).astype(np.uint8)
    return S, st


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("variant", ["no-autoreset", "continue-undefined", "uploaded", "mapped"])
def test_step_rewards_variants(pb, orc, teams, variant):
    """without AUTORESET (frozen envs get zeros), with CONTINUE_UNDEFINED, on uploaded done / invalid / inconsistent
    states, and with page-locked mapped host buffers"""
    n, ticks = 4099, 60
    a = pb.Batch(n, n_templates=64, max_ticks=40, teams=teams)
    c = pb.Batch(n, n_templates=64, max_ticks=40, teams=teams)
    flags = {"no-autoreset": pb.STEP_COUNT, "continue-undefined": pb.STEP_AUTORESET | pb.STEP_COUNT | pb.STEP_CONTINUE_UNDEFINED,
             "uploaded": pb.STEP_AUTORESET | pb.STEP_COUNT, "mapped": pb.STEP_AUTORESET | pb.STEP_COUNT}[variant]
    if variant == "uploaded":
        S, st = _uploaded(pb, orc, n, teams, 41 + teams)
        a.upload(S, st)
        c.upload(S, st)
    counts = _drive(pb, a, c, teams, ticks, flags, 23, simple=variant == "mapped", mapped=variant == "mapped")
    assert counts[1] > 0 and counts[2] > 0, counts
    if variant == "no-autoreset":
        assert c.stats().episodes == 0 and (c.status() & DONE).any()
    a.close(); c.close()


@pytest.mark.gpu
def test_step_rewards_refusals(pb, monkeypatch):
    """POM_E_ARG, with nothing stepped: RAW, OVERLAP and unknown flags, null rewards or moves, pageable buffers, a
    misaligned rewards buffer, a handle made with POM_STEP_KERNEL=tile"""
    n = 300
    b = pb.Batch(n, n_templates=8)
    L = pb.lib()
    mv, rw, st = b.alloc(4 * n), b.alloc(4 * n), b.alloc(n)
    b.generate_moves(mv, 1, 0, 6)
    S0, s0 = b.download()
    page = np.zeros(4 * n, np.int8)
    pp = page.ctypes.data_as(C.c_void_p)
    for f in (pb.STEP_RAW, pb.STEP_OVERLAP, pb.STEP_AUTORESET | pb.STEP_RAW, 0x40000000, 0x20):
        assert L.pom_batch_step_rewards(b.h, mv, f, rw, st) == -1, f
    assert L.pom_batch_step_rewards(b.h, mv, 0, None, st) == -1
    assert L.pom_batch_step_rewards(b.h, None, 0, rw, st) == -1
    assert L.pom_batch_step_rewards(b.h, mv, 0, pp, st) == -1
    assert L.pom_batch_step_rewards(b.h, pp, 0, rw, st) == -1
    assert L.pom_batch_step_rewards(b.h, mv, 0, rw, pp) == -1
    assert L.pom_batch_step_rewards(b.h, mv, 0, C.c_void_p(rw.value + 1), st) == -1 and b"aligned" in L.pom_last_error()
    assert L.pom_batch_step_rewards(None, mv, 0, rw, st) == -1
    S1, s1 = b.download()
    assert S1.tobytes() == S0.tobytes() and (s1 == s0).all() and b.stats().env_steps == 0
    assert L.pom_batch_step_rewards(b.h, mv, pb.STEP_COUNT, rw, None) == 0
    b.sync()
    assert b.stats().env_steps == n
    monkeypatch.setenv("POM_STEP_KERNEL", "tile")
    t = pb.Batch(n, n_templates=8)
    monkeypatch.delenv("POM_STEP_KERNEL")
    assert L.pom_batch_step_rewards(t.h, mv, 0, rw, st) == -1 and b"POM_STEP_KERNEL" in L.pom_last_error()
    for p in (mv, rw, st):
        b.free(p)
    b.close(); t.close()


BATCH_ENV_CPP = r"""
#include <cstdio>
#include <cstring>
#include <vector>
#include "pom_bboard.hpp"
using namespace bboard;
int main()
{
    const size_t n = 4096;
    BatchEnvironment env(n, 0, 0, 64, 0x1337, 0, TEAMS), plain(n, 0, 0, 64, 0x1337, 0, TEAMS), raw(n, 0, 0, 64, 0x1337, 0, TEAMS);
    void* pinned = nullptr;
    if(pom_host_alloc(9 * n, &pinned) != POM_OK) return 1;
    uint8_t* m8 = static_cast<uint8_t*>(pinned);
    int8_t* rw_raw = reinterpret_cast<int8_t*>(m8 + 4 * n);
    uint8_t* st_raw = m8 + 8 * n;
    std::vector<Move> mv(4 * n);
    std::vector<int8_t> rw(4 * n);
    long plus = 0, minus = 0;
    for(uint32_t t = 0; t < 300; t++)
    {
        for(size_t e = 0; e < n; e++)
        {
            const uint32_t m = pom_rng_moves(5, e, t, 6);
            for(int a = 0; a < 4; a++) { mv[4 * e + a] = Move((m >> (8 * a)) & 0xFF); m8[4 * e + a] = uint8_t((m >> (8 * a)) & 0xFF); }
        }
        const size_t running = env.Step(mv.data(), rw.data());
        if(running != plain.Step(mv.data())) return 2;
        if(pom_batch_step_rewards(raw.Handle(), m8, 0, rw_raw, st_raw) != POM_OK || pom_batch_sync(raw.Handle()) != POM_OK) return 3;
        if(std::memcmp(rw.data(), rw_raw, 4 * n) != 0) return 4;
        for(size_t i = 0; i < n; i++) if(env.Status()[i] != st_raw[i] || plain.Status()[i] != st_raw[i]) return 5;
        for(size_t i = 0; i < 4 * n; i++) { plus += rw[i] == 1; minus += rw[i] == -1; }
    }
    const std::vector<State> a = env.States(), b = plain.States();
    for(size_t i = 0; i < n; i++) if(std::memcmp(&a[i], &b[i], sizeof(State)) != 0) return 6;
    pom_host_free(pinned);
    std::printf("%ld %ld\n", plus, minus);
    return 0;
}
"""


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
def test_batch_environment_step_with_rewards(pb, tmp_path, teams):
    """bboard::BatchEnvironment::Step(moves, rewards) == Step(moves) for states, status bytes and running count, and its
    rewards == pom_batch_step_rewards on a third handle"""
    src, exe = tmp_path / "rewards_env.cpp", tmp_path / "rewards_env"
    src.write_text(BATCH_ENV_CPP.replace("TEAMS", "true" if teams else "false"))
    lib = os.path.join(ROOT, "pomcpp_b200")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                          os.path.join(lib, "host", "libpom_host.a"), "-L" + lib, "-lpom_b200", "-Wl,-rpath," + lib],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    plus, minus = map(int, run.stdout.split())
    assert plus > 0 and minus > 0
