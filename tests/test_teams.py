"""The 2v2 team game (POM_INIT_TEAMS): team 0 = agents 0 and 2, team 1 = agents 1 and 3.  The reference has no team mode,
so this file holds the definition (TeamRestatement: the episode rule on top of the restatement's bare Step, and the
restatement's SimpleAgent with the teammate hidden from its enemy searches) and pins the device code to it:
  CPU  the team instantiation of the kernel body built for the host (tests/teamsim) == the definition, tick by tick, on
       random, harmless, stress and inconsistent states; explicit cases of the rule; the team-aware SimpleAgent; the
       coupling of a team game and a free-for-all game driven with the same moves.
  GPU  every entry point on a team handle == the definition, every field and status byte, with the episode counters."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle

DONE, DRAW, INVALID, TRUNC = 0x01, 0x02, 0x10, 0x20


class TeamRestatement:
    """The team game on the restatement (oracle/pom_oracle.c, pom_oracle_agent.c), which is free-for-all:
      env_step_batch    Environment::Step with the team rule: bare Step (pom_oracle_step), timeStep++, then a team is
                        alive while one of its agents' dead flags is clear (not the aliveAgents counter): none alive ->
                        DONE | DRAW, one -> DONE with the team index in the winner field; INVALID as in free-for-all
      simple_*          the SimpleAgent of agent a acting on the state with its teammate a ^ 2 marked dead: the agent reads
                        the other agents' dead flags only in IsAdjacentEnemy and MoveTowardsEnemy (strategy.cpp:165-183,
                        296-312), so this is "the teammate is no enemy" and nothing else; the board is left as it is
    Everything else is the restatement's."""

    def __init__(self, orc):
        self.o = orc

    def __getattr__(self, name):
        return getattr(self.o, name)

    def env_step_batch(self, S, status, moves, flags=None):
        live = np.nonzero((status & (DONE | INVALID)) == 0)[0]
        sub = S[live]
        f = np.zeros(live.shape[0], np.uint8)
        self.o.step_batch(sub, np.ascontiguousarray(moves[live]), f)
        sub["timeStep"] += 1
        S[live] = sub
        dead = sub["agents"]["dead"] != 0
        a0, a1 = ~dead[:, 0] | ~dead[:, 2], ~dead[:, 1] | ~dead[:, 3]
        st = status[live].astype(np.int64)
        ended = (st & INVALID) | DONE
        st = np.where(~a0 & ~a1, ended | DRAW, np.where(a0 != a1, ended | (np.where(a0, 0, 1) << 2), st))
        st[(f & 0x3E) != 0] |= INVALID                       # POM_ORC_INVALID_MASK: left the reference's domain
        status[live] = st.astype(np.uint8)
        if flags is not None:
            flags[:] = 0
            flags[live] = f

    @staticmethod
    def _hide_teammate(S, a):
        V = S.copy()
        V["agents"]["dead"][:, a ^ 2] = 1
        return V

    def simple_moves_batch(self, S, status, A, seed, env0, tick, agent_mask, moves):
        for a in range(4):
            if (agent_mask >> a) & 1:
                self.o.simple_moves_batch(self._hide_teammate(S, a), status, A, seed, env0, tick, 1 << a, moves)

    def simple_act(self, s, agent_id, st, draw):
        return self.o.simple_act(self._hide_teammate(s, agent_id), agent_id, st, draw)

    def is_adjacent_enemy(self, s, agent_id, dist):
        return self.o.is_adjacent_enemy(self._hide_teammate(s, agent_id), agent_id, dist)

    def move_towards(self, s, agent_id, kind, a, b=0):
        return self.o.move_towards(self._hide_teammate(s, agent_id), agent_id, kind, a, b)


class TeamSim:
    """tests/teamsim: the TEAMS instantiation of the device code built for the host; records packed by tests/hostsim"""

    def __init__(self, so):
        from hostsim import HostSim
        self.h = HostSim()
        L = self.lib = C.CDLL(so)
        vp = C.c_void_p
        L.teamsim_step_records.argtypes = [vp, C.c_long, vp, C.c_int, vp]
        L.teamsim_simple_moves.argtypes = [vp, C.c_long, vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, vp]
        self.by_rays = False

    def set_by_rays(self, on):
        self.by_rays = bool(on)

    def pack(self, S, status=None):
        return self.h.pack(S, status)

    def unpack(self, recs):
        return self.h.unpack(recs)

    def step_records(self, recs, moves):
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.teamsim_step_records(p(recs), recs.shape[0], p(moves), int(self.by_rays), None)

    def simple_moves(self, recs, A, seed, env0, tick, mask, moves):
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.teamsim_simple_moves(p(recs), recs.shape[0], p(A), seed, env0, tick, mask, p(moves))


@pytest.fixture
def team_orc(orc):
    return TeamRestatement(orc)


@pytest.fixture(scope="module")
def teamsim_so(tmp_path_factory):
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    so = str(tmp_path_factory.mktemp("teamsim") / "libteamsim.so")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-I", os.path.join(root, "include"),
                          "-I", os.path.join(root, "pomcpp_b200", "csrc"), "-o", so, os.path.join(here, "teamsim", "teamsim.cpp")],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return so


@pytest.fixture
def hs(teamsim_so):
    return TeamSim(teamsim_so)


def _games(orc, n, stress=False, seed=0):
    """n games from InitState on clean seeds; stress: kicks, several bombs, long flames (more deaths)"""
    seeds = oracle.clean_seeds(128)
    S = orc.zero_state(n)
    for e in range(n):
        assert orc.init_state(S[e:e + 1], seeds[e % len(seeds)]) == 0
    if stress:
        rng = np.random.default_rng(seed)
        S["agents"]["canKick"] = rng.integers(0, 2, (n, 4))
        S["agents"]["maxBombCount"] = rng.integers(1, 5, (n, 4))
        S["agents"]["bombStrength"] = rng.integers(1, 4, (n, 4))
    return S


def _outcomes(status):
    """counts of (team 0 won, team 1 won, draws) among finished, valid envs"""
    fin = (status & (DONE | INVALID)) == DONE
    won = fin & ((status & DRAW) == 0)
    w = (status >> 2) & 3
    return int((won & (w == 0)).sum()), int((won & (w == 1)).sum()), int((fin & ((status & DRAW) != 0)).sum())


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("by_rays", [False, True], ids=["one-lane", "by-rays"])
@pytest.mark.parametrize("kind", ["random", "harmless", "stress"])
def test_kernel_body_team_rule_matches_oracle(team_orc, hs, kind, by_rays):
    """every field and the whole status byte after every tick; finished games restart from their first state"""
    orc = team_orc
    hs.set_by_rays(by_rays)
    n, ticks, nact = 1024, 260, 5 if kind == "harmless" else 6
    S = _games(orc, n, stress=kind == "stress", seed=11)
    recs, bad = hs.pack(S)
    assert not bad.any()
    S0, recs0 = S.copy(), recs.copy()
    st = np.zeros(n, np.uint8)
    totals = np.zeros(3, np.int64)
    for t in range(ticks):
        mv = orc.rng_moves(2101, 0, n, t, nact)
        orc.env_step_batch(S, st, mv)
        hs.step_records(recs, mv)
        G, gst = hs.unpack(recs)
        e, why = orc.diff_batch(G, S)
        assert e == -1, "tick %d env %d field group %d" % (t, e, why)
        assert (gst == st).all(), "status differs at tick %d (env %d)" % (t, np.nonzero(gst != st)[0][0])
        totals += _outcomes(st)
        idx = np.nonzero(st & (DONE | INVALID))[0]
        S[idx], recs[idx], st[idx] = S0[idx], recs0[idx], 0
    if kind != "harmless":
        assert (totals > 0).all(), totals                      # both teams won somewhere, and some games were drawn


@pytest.mark.parametrize("seed", [501, 502])
def test_team_rule_on_inconsistent_states(team_orc, hs, seed):
    """uploaded states no game reaches (tests/test_fuzz_states.py), plus an aliveAgents counter out of step with the dead
    flags in a third of them: the flags decide"""
    from test_fuzz_states import mutated_states
    orc = team_orc
    S = mutated_states(orc, seed, 3000)
    rng = np.random.default_rng(seed)
    off = rng.random(S.shape[0]) < 0.33
    S["aliveAgents"][off] = rng.integers(0, 5, int(off.sum()))
    recs, bad = hs.pack(S, np.zeros(S.shape[0], np.uint8))
    S, recs = S[bad == 0].copy(), recs[bad == 0].copy()
    n = S.shape[0]
    assert n > 1500
    st = np.zeros(n, np.uint8)
    for t in range(12):
        mv = orc.rng_moves(seed + 1000, 0, n, t, 6)
        orc.env_step_batch(S, st, mv)
        hs.step_records(recs, mv)
        G, gst = hs.unpack(recs)
        invalid = (st & INVALID) != 0
        e, why = orc.diff_batch(G, S, invalid.astype(np.uint8))
        assert e == -1, "tick %d env %d field group %d" % (t, e, why)
        assert ((gst & (DONE | INVALID)) == (st & (DONE | INVALID))).all()
        assert (gst[~invalid] == st[~invalid]).all(), "tick %d" % t
    assert (st & DONE).any()


# (agents killed, aliveAgents forced to, status after one quiet tick in the team game, and in free-for-all)
RULE_CASES = [
    ((0, 2), None, DONE | (1 << 2), 0),
    ((1, 3), None, DONE | (0 << 2), 0),
    ((0, 1), None, 0, 0),
    ((3,), None, 0, 0),
    ((0, 1, 2, 3), None, DONE | DRAW, DONE | DRAW),
    ((0, 1, 2), None, DONE | (1 << 2), DONE | (3 << 2)),
    ((1, 3), 3, DONE | (0 << 2), 0),                # the counter disagrees with the flags: the flags decide
    ((), 0, 0, DONE | DRAW),
    ((0, 2), 1, DONE | (1 << 2), DONE | (3 << 2)),
]


@pytest.mark.parametrize("killed,alive,want_team,want_ffa", RULE_CASES)
def test_team_rule_cases(team_orc, hs, killed, alive, want_team, want_ffa):
    orc = team_orc
    S = _games(orc, 1)
    orc.kill(S, *killed)
    if alive is not None:
        S["aliveAgents"][0] = alive
    recs, bad = hs.pack(S)
    assert not bad.any()
    idle = np.zeros((1, 4), np.uint8)
    T, st = S.copy(), np.zeros(1, np.uint8)
    orc.env_step_batch(T, st, idle)
    assert st[0] == want_team
    hs.step_records(recs, idle)
    assert hs.unpack(recs)[1][0] == want_team
    F, sf = S.copy(), np.zeros(1, np.uint8)
    orc.o.env_step_batch(F, sf, idle)
    assert sf[0] == want_ffa


def _mid_game(orc, n, seed):
    """agents spread over the board by 60 harmless random ticks"""
    S = _games(orc, n)
    st = np.zeros(n, np.uint8)
    for t in range(60):
        orc.env_step_batch(S, st, orc.rng_moves(seed, 0, n, t, 5))
    return S


@pytest.mark.parametrize("states", ["mid-game", "inconsistent"])
def test_team_simple_agent_matches_oracle(team_orc, hs, states):
    """the device SimpleAgent in team mode (host build) == the restatement: moves and memories, act after act, with the
    games stepped under the team rule in between; and the team agent does play differently from the free-for-all one"""
    from test_fuzz_states import mutated_states
    orc = team_orc
    S = _mid_game(orc, 2000, 7) if states == "mid-game" else mutated_states(orc, 403, 3000)
    recs, bad = hs.pack(S, np.zeros(S.shape[0], np.uint8))
    S, recs = S[bad == 0].copy(), recs[bad == 0].copy()
    n = S.shape[0]
    st = np.zeros(n, np.uint8)
    A = orc.simple_agents(n)
    B = A.copy()
    spared = 0
    for t in range(16):
        ffa = np.zeros((n, 4), np.uint8)
        orc.o.simple_moves_batch(S, st, A.copy(), 9, 0, t, 15, ffa)
        mv, mv2 = np.zeros((n, 4), np.uint8), np.zeros((n, 4), np.uint8)
        orc.simple_moves_batch(S, st, A, 9, 0, t, 15, mv)
        hs.simple_moves(recs, B, 9, 0, t, 15, mv2)
        live = (st & (DONE | INVALID)) == 0
        assert (mv[live] == mv2[live]).all(), "act %d env %d" % (t, np.nonzero((mv != mv2).any(1) & live)[0][0])
        assert A.tobytes() == B.tobytes(), "memories after act %d" % t
        spared += int((mv != ffa).any(1)[live].sum())
        orc.env_step_batch(S, st, mv)
        hs.step_records(recs, mv)
        invalid = (st & INVALID) != 0
        assert orc.diff_batch(hs.unpack(recs)[0], S, invalid.astype(np.uint8))[0] == -1
    assert spared > 100, spared                                 # the team agent does spare its teammate


def _duel(orc, teammate_at):
    """agent 0 at (5, 5), its teammate 2 at `teammate_at`, the enemies 1 and 3 in far corners; open board"""
    S = orc.zero_state()
    orc.put_agent(S, 5, 5, 0)
    orc.put_agent(S, *teammate_at, 2)
    orc.put_agent(S, 0, 0, 1)
    orc.put_agent(S, 10, 10, 3)
    return S


def test_simple_agent_never_targets_its_teammate(team_orc, hs):
    """IsAdjacentEnemy (bomb at distance 1, hunt within 7) and MoveTowardsEnemy skip the teammate in a team game"""
    orc = team_orc
    near, mid = _duel(orc, (5, 6)), _duel(orc, (5, 8))
    assert not orc.is_adjacent_enemy(near, 0, 1) and not orc.is_adjacent_enemy(mid, 0, 7)
    assert orc.move_towards(mid, 0, 2, 7) == 0                  # no enemy within 7: IDLE
    # the agent's memory holds four distinct recent positions: no _HasRPLoop, so a hunt would walk towards the target
    mem = orc.simple_agents(1)
    mem["recent"][0, 0] = [0x11, 0x12, 0x13, 0x14]
    mem["rp_count"][0, 0] = 4
    team_moves = {"near": set(), "mid": set()}
    for name, S in (("near", near), ("mid", mid)):
        recs, bad = hs.pack(S)
        assert not bad.any()
        for t in range(12):
            A, B = mem.copy(), mem.copy()
            mv, mv2 = np.zeros((1, 4), np.uint8), np.zeros((1, 4), np.uint8)
            orc.simple_moves_batch(S, None, A, 3, 0, t, 1, mv)
            hs.simple_moves(recs, B, 3, 0, t, 1, mv2)
            assert mv[0, 0] == mv2[0, 0] and A.tobytes() == B.tobytes()
            team_moves[name].add(int(mv[0, 0]))
    assert 5 not in team_moves["near"]                          # no BOMB for a teammate next door
    assert len(team_moves["mid"]) > 1                           # random safe steps, not a walk towards the teammate
    ffa = orc.o
    assert ffa.is_adjacent_enemy(near, 0, 1) and ffa.move_towards(mid, 0, 2, 7) == 2
    for t in range(12):
        A = mem.copy()
        for S, want in ((near, 5), (mid, 2)):                  # free-for-all: BOMB the neighbour, walk DOWN to the other
            mv = np.zeros((1, 4), np.uint8)
            ffa.simple_moves_batch(S, None, A.copy(), 3, 0, t, 1, mv)
            assert mv[0, 0] == want


def _coupling(ticks, step_ffa, step_team):
    """A team game and a free-for-all game from the same InitState, driven with the same moves, no reset.  step_*(t)
    runs tick t and returns (states, status bytes).  Checks, per env:
      - the team game ends no later than the free-for-all game;
      - up to (and at) the tick it ends, its state is the free-for-all game's;
      - a free-for-all win by agent w is a win of team w & 1, a team draw happens only at the tick of a free-for-all draw.
    Returns (team games that ended strictly earlier, team wins, team draws)."""
    end_t = end_f = None
    for t in range(ticks):
        F, sf = step_ffa(t)
        T, stt = step_team(t)
        if end_t is None:
            end_t = np.full(sf.shape[0], -1)
            end_f = np.full(sf.shape[0], -1)
            win_t, win_f = np.zeros(sf.shape[0], np.uint8), np.zeros(sf.shape[0], np.uint8)
        running = end_t < 0
        assert oracle.restatement().diff_batch(T[running], F[running])[0] == -1, "tick %d" % t
        assert ((stt[running] & INVALID) == (sf[running] & INVALID)).all()
        newt = running & ((stt & DONE) != 0)
        newf = (end_f < 0) & ((sf & DONE) != 0)
        end_t[newt], win_t[newt] = t, stt[newt]
        end_f[newf], win_f[newf] = t, sf[newf]
    valid = ((win_t | win_f) & INVALID) == 0
    ff = valid & (end_f >= 0)
    assert (end_t[ff] >= 0).all() and (end_t[ff] <= end_f[ff]).all()
    fwin = ff & ((win_f & DRAW) == 0)
    assert ((win_t[fwin] & DRAW) == 0).all() and (((win_t[fwin] >> 2) & 3) == ((win_f[fwin] >> 2) & 1)).all()
    tdraw = valid & (end_t >= 0) & ((win_t & DRAW) != 0)
    assert (end_f[tdraw] == end_t[tdraw]).all() and ((win_f[tdraw] & DRAW) != 0).all()
    earlier = valid & (end_t >= 0) & ((end_f < 0) | (end_t < end_f))
    return int(earlier.sum()), int((valid & (end_t >= 0) & ((win_t & DRAW) == 0)).sum()), int(tdraw.sum())


def test_team_game_couples_with_free_for_all(orc):
    n, ticks, seed = 1500, 400, 61
    F = _games(orc, n, stress=True, seed=3)
    T = F.copy()
    sf, stt = np.zeros(n, np.uint8), np.zeros(n, np.uint8)

    def step(S, st, game):
        def run(t):
            game.env_step_batch(S, st, orc.rng_moves(seed, 0, n, t, 6))
            return S, st
        return run
    earlier, wins, draws = _coupling(ticks, step(F, sf, orc), step(T, stt, TeamRestatement(orc)))
    assert earlier > 50 and wins > 50 and draws > 0, (earlier, wins, draws)


# ----------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


class OracleRun:
    """the restatement replaying a per-tick loop with pom_batch_step's episode rule: step, truncate at max_ticks, count,
    reset to template[(env_offset + e + episode) % n_templates] (when auto-resetting)"""

    def __init__(self, orc, S, T, env0=0, max_ticks=0):
        self.o, self.S, self.T, self.env0, self.max_ticks = orc, S, T, env0, max_ticks
        n = S.shape[0]
        self.status = np.zeros(n, np.uint8)
        self.episode = np.zeros(n, np.int64)
        self.stats = np.zeros(10, np.int64)

    def tick(self, mv, autoreset=True, count=True):
        """returns every env's end-of-tick status byte (before the reset: what status_out reports)"""
        S, st = self.S, self.status
        live = (st & (DONE | INVALID)) == 0
        if count:
            self.stats[0] += int(live.sum())
        self.o.env_step_batch(S, st, np.ascontiguousarray(mv))
        if not autoreset:
            return st.copy()
        if self.max_ticks:
            st[live & ((st & DONE) == 0) & (S["timeStep"] >= self.max_ticks)] |= TRUNC
        end = st.copy()
        for e in np.nonzero(live & ((st & (DONE | INVALID | TRUNC)) != 0))[0]:
            s = self.stats
            s[1] += 1
            if st[e] & DONE:
                s[6 if st[e] & DRAW else 2 + ((st[e] >> 2) & 3)] += 1
            elif st[e] & TRUNC:
                s[7] += 1
            else:
                s[9] += 1
            s[8] += int(S["timeStep"][e])
            self.episode[e] += 1
            S[e] = self.T[(self.env0 + e + self.episode[e]) % self.T.shape[0]]
            st[e] = 0
        return end


def _check_stats(b, want=None):
    s = b.stats()
    assert s.wins[2] == 0 and s.wins[3] == 0
    assert s.episodes == s.wins[0] + s.wins[1] + s.draws + s.truncated + s.invalid
    if want is not None:
        assert (s.as_array() == want).all(), (s.as_dict(), want)
    return s


@pytest.mark.gpu
def test_team_handle_reports_its_mode(pb):
    a, c = pb.Batch(64, n_templates=4), pb.Batch(64, n_templates=4, teams=True)
    assert not a.teams() and c.teams()
    assert pb.lib().pom_batch_teams(None) == -1
    a.close(); c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["step", "tile", "step_host", "step_host_pinned", "step_host_async"])
def test_team_per_tick_step_matches_oracle(pb, team_orc, path, monkeypatch):
    """pom_batch_step (persistent and tile kernel), _step_host (pageable and pinned), _step_host_async with auto-reset,
    truncation and counters: states and status bytes every tick, counters at the end"""
    n, ticks, seed, env0 = 3000 + 17, 90, 303, 40
    if path == "tile":
        monkeypatch.setenv("POM_STEP_KERNEL", "tile")
    b = pb.Batch(n, env_offset=env0, n_templates=64, max_ticks=50, teams=True)
    monkeypatch.delenv("POM_STEP_KERNEL", raising=False)
    T, _ = b.templates()
    S, _ = b.download()
    R = OracleRun(team_orc, S, T, env0, 50)
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT
    dev = b.alloc(4 * n)
    mvp = stp = None
    if path in ("step_host_pinned", "step_host_async"):
        mvp, o1 = pb.pinned_array((n, 4), np.uint8)
        stp, o2 = pb.pinned_array((n,), np.uint8)
    out = np.zeros(n, np.uint8)
    for t in range(ticks):
        mv = team_orc.rng_moves(seed, env0, n, t, 6)
        if path in ("step", "tile"):
            b.generate_moves(dev, seed, t, 6)
            b.step(dev, flags)
            got = None
        elif path == "step_host":
            b.step_host(mv, out, flags)
            got = out
        else:
            mvp[:] = mv
            (b.step_host if path == "step_host_pinned" else b.step_host_async)(mvp, stp, flags)
            b.sync()
            got = stp
        end = R.tick(mv)
        if got is not None:
            assert (got == end).all(), "tick %d env %d" % (t, np.nonzero(got != end)[0][0])
        if t % 15 == 14 or t == ticks - 1:
            G, gst = b.download()
            assert team_orc.diff_batch(G, S)[0] == -1 and (gst == R.status).all(), "tick %d" % t
    s = _check_stats(b, R.stats)
    assert s.wins[0] > 0 and s.wins[1] > 0 and s.truncated > 0
    b.free(dev)
    if mvp is not None:
        pb.pinned_free(o1); pb.pinned_free(o2)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fused_kernel", [0, 1])
def test_team_step_compact_and_step_observe(pb, team_orc, fused_kernel, monkeypatch):
    """pom_batch_step_compact (joint actions in, done bits and finished-env list out, planes) and pom_batch_step_observe,
    both forms of the planes (observe kernel behind the step, POM_OBS_FUSED=1: written by the step kernel)"""
    n, ticks, env0 = 4099, 40, 0
    monkeypatch.setenv("POM_OBS_FUSED", str(fused_kernel))
    a = pb.Batch(n, n_templates=64, max_ticks=30, teams=True)
    c = pb.Batch(n, n_templates=64, max_ticks=30, teams=True)
    monkeypatch.delenv("POM_OBS_FUSED")
    T, _ = a.templates()
    Sa, _ = a.download()
    Sc = Sa.copy()
    Ra, Rc = OracleRun(team_orc, Sa, T, env0, 30), OracleRun(team_orc, Sc, T, env0, 30)
    stride = int(pb.lib().pom_batch_obs_stride(a.h))
    obs_a, obs_c = a.alloc(2 * stride * pb.OBS_BYTES), c.alloc(stride * pb.OBS_BYTES)
    joint, o1 = pb.pinned_array((n,), np.uint16)
    bits, o2 = pb.pinned_array(((n + 31) // 32,), np.uint32)
    fenv, o3 = pb.pinned_array((n,), np.uint32)
    fst, o4 = pb.pinned_array((n,), np.uint8)
    fcnt, o5 = pb.pinned_array((1,), np.uint32)
    mv_dev = c.alloc(4 * n)
    rng = np.random.default_rng(8)
    flags = pb.STEP_AUTORESET | pb.STEP_COUNT
    ended_total = 0
    for t in range(ticks):
        mv = rng.integers(0, 6, (n, 4), dtype=np.uint8)
        joint[:] = pb.joint_of_moves(mv)
        a.step_compact(joint, bits, fenv, fst, fcnt, flags, obs_dev=obs_a, obs_agent_mask=0b0101, obs_view=4)
        pb.lib().pom_device_copy(0, mv_dev, mv.ctypes.data_as(C.c_void_p), 4 * n)
        c.step_observe(mv_dev, obs_c, 0b0010, 3, flags)
        a.sync(); c.sync()
        end = Ra.tick(mv)
        Rc.tick(mv)
        ended = (end & (DONE | TRUNC | INVALID)) != 0
        got_bits = np.unpackbits(bits.view(np.uint8), bitorder="little")[:n].astype(bool)
        assert (got_bits == ended).all(), "done bits, tick %d" % t
        k = int(fcnt[0])
        order = np.argsort(fenv[:k])
        assert k == int(ended.sum()) and (fenv[:k][order] == np.nonzero(ended)[0]).all() and (fst[:k][order] == end[ended]).all()
        ended_total += k
        if t % 10 == 9:
            for b, R, obs, agents, view in ((a, Ra, obs_a, (0, 2), 4), (c, Rc, obs_c, (1,), 3)):
                G, gst = b.download()
                assert team_orc.diff_batch(G, R.S)[0] == -1 and (gst == R.status).all(), "tick %d" % t
                got = np.zeros((len(agents), stride, pb.OBS_BYTES), np.uint8)
                pb.lib().pom_device_copy(0, got.ctypes.data_as(C.c_void_p), obs, got.nbytes)
                for j, ag in enumerate(agents):
                    assert (got[j, :n] == team_orc.observe_planes_batch(R.S, ag, view)).all(), "agent %d tick %d" % (ag, t)
    assert ended_total > 500
    _check_stats(a, Ra.stats)
    _check_stats(c, Rc.stats)
    a.free(obs_a); c.free(obs_c); c.free(mv_dev)
    for o in (o1, o2, o3, o4, o5):
        pb.pinned_free(o)
    a.close(); c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("harmless,no_reset", [(0, False), (1, False), (0, True)])
def test_team_rollout_matches_oracle(pb, team_orc, harmless, no_reset):
    """the fused rollout with random / harmless agents (the team game runs the generic image: there is no SPEC one)"""
    from test_gpu_parity import _oracle_rollout
    n, ticks, seed, env0 = 2048 + 5, 150, 71, 900
    b = pb.Batch(n, env_offset=env0, n_templates=64, max_ticks=100, teams=True)
    T, _ = b.templates()
    S, _ = b.download()
    flags = (pb.ROLL_HARMLESS if harmless else 0) | (pb.ROLL_NO_RESET if no_reset else 0)
    b.rollout(100, seed, 0, flags)
    b.rollout(ticks - 100, seed, 100, flags)
    G, gst = b.download()
    status, stats = _oracle_rollout(team_orc, S, T, env0, ticks, seed, 5 if harmless else 6, 100, no_reset=no_reset)
    e, why = team_orc.diff_batch(G, S)
    assert e == -1, "env %d field group %d" % (e, why)
    assert (gst == status).all()
    _check_stats(b, stats)
    b.close()


@pytest.mark.gpu
def test_team_step_seq_matches_oracle(pb, team_orc):
    n, ticks = 1500, 70
    b = pb.Batch(n, n_templates=32, max_ticks=45, teams=True)
    T, _ = b.templates()
    S, _ = b.download()
    R = OracleRun(team_orc, S, T, 0, 45)
    mv = np.random.default_rng(4).integers(0, 6, (ticks, n, 4), dtype=np.uint8)
    dev = b.alloc(mv.nbytes)
    pb.lib().pom_device_copy(0, dev, mv.ctypes.data_as(C.c_void_p), mv.nbytes)
    b.step_seq(dev, ticks)
    for t in range(ticks):
        R.tick(mv[t])
    G, gst = b.download()
    assert team_orc.diff_batch(G, S)[0] == -1 and (gst == R.status).all()
    _check_stats(b, R.stats)
    b.free(dev)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mask,harmless,max_ticks,no_reset", [(15, 0, 800, False), (0b0101, 1, 90, False),
                                                               (0b1011, 0, 0, True)])
def test_team_rollout_with_simple_agents_matches_oracle(pb, team_orc, mask, harmless, max_ticks, no_reset):
    """the fused rollout with team-aware SimpleAgents (k_rollout with the policy)"""
    from test_gpu_policy import _oracle_policy_rollout
    n, ticks, seed, env0 = 1024 + 33, 220, 808, 5000
    b = pb.Batch(n, env_offset=env0, n_templates=40, max_ticks=max_ticks, teams=True)
    T, _ = b.templates()
    S, _ = b.download()
    A = team_orc.simple_agents(n)
    flags = pb.ROLL_SIMPLE(mask) | (pb.ROLL_HARMLESS if harmless else 0) | (pb.ROLL_NO_RESET if no_reset else 0)
    b.rollout(100, seed, 0, flags)
    b.rollout(ticks - 100, seed, 100, flags)
    G, gst = b.download()
    status, stats = _oracle_policy_rollout(team_orc, S, T, A, env0, ticks, seed, 5 if harmless else 6, max_ticks, mask,
                                           no_reset=no_reset)
    e, why = team_orc.diff_batch(G, S)
    assert e == -1, "env %d field group %d" % (e, why)
    assert (gst == status).all()
    _check_stats(b, stats)
    assert b.policy_download().tobytes() == A.tobytes()
    b.close()


@pytest.mark.gpu
def test_team_rollout_with_simple_agents_tick_by_tick(pb, team_orc, monkeypatch):
    """a large batch with SimpleAgents runs k_policy_moves + the per-tick step kernel (FREEZE image) tick by tick; the
    same as the fused kernel (POM_ROLL_POLICY=fused) and, on a slice replayed by the restatement, as the definition"""
    from test_gpu_policy import _oracle_policy_rollout
    n, ticks, seed = (1 << 16) + 4099, 45, 77
    monkeypatch.setenv("POM_ROLL_POLICY", "fused")
    a = pb.Batch(n, n_templates=128, max_ticks=60, teams=True)
    monkeypatch.delenv("POM_ROLL_POLICY")
    c = pb.Batch(n, n_templates=128, max_ticks=60, teams=True)
    T, _ = c.templates()
    for x in (a, c):
        l0 = x.launch_count()
        x.rollout(ticks, seed, 0, pb.ROLL_SIMPLE(0b1011))
        x.launches = x.launch_count() - l0
    assert a.launches == 1 and c.launches == 2 * ticks
    A, sa = a.download()
    Cc, sc = c.download()
    assert A.tobytes() == Cc.tobytes() and (sa == sc).all()
    assert a.stats().as_dict() == c.stats().as_dict()
    _check_stats(c)
    lo, cnt = 40_001, 256
    S = np.stack([T[(lo + e) % 128] for e in range(cnt)]).astype(oracle.STATE_DT)
    M = team_orc.simple_agents(cnt)
    status, _ = _oracle_policy_rollout(team_orc, S, T, M, lo, ticks, seed, 6, 60, 0b1011)
    assert team_orc.diff_batch(Cc[lo:lo + cnt], S)[0] == -1 and (sc[lo:lo + cnt] == status).all()
    assert c.policy_download(lo, cnt).tobytes() == M.tobytes()
    a.close(); c.close()


@pytest.mark.gpu
def test_team_policy_entry_points_match_oracle(pb, team_orc):
    """pom_batch_policy_moves (device buffer), _policy_moves_host and _policy_act on a team handle"""
    n, seed = 1200, 21
    b = pb.Batch(n, n_templates=48, teams=True)
    b.rollout(30, 3, 0, pb.ROLL_NO_RESET)
    S, status = b.download()
    A = team_orc.simple_agents(n)
    dev = b.alloc(4 * n)
    for t in range(30):
        mv = team_orc.rng_moves(seed, 0, n, t, 6)
        want = mv.copy()
        team_orc.simple_moves_batch(S, status, A, seed, 0, t, 0b0111, want)
        live = (status & (DONE | INVALID)) == 0
        if t % 2:
            got = mv.copy()
            b.policy_moves_host(got, seed, t, 0b0111)
        else:
            pb.lib().pom_device_copy(0, dev, mv.ctypes.data_as(C.c_void_p), 4 * n)
            b.policy_moves(dev, seed, t, 0b0111)
            b.sync()
            got = np.zeros((n, 4), np.uint8)
            pb.lib().pom_device_copy(0, got.ctypes.data_as(C.c_void_p), dev, 4 * n)
        assert (got[live] == want[live]).all(), "tick %d" % t
        b.step_host(got, None, 0)
        team_orc.env_step_batch(S, status, want)
    assert b.policy_download().tobytes() == A.tobytes()
    G, gst = b.download()
    assert team_orc.diff_batch(G, S)[0] == -1 and (gst == status).all()
    # one agent at a time with the caller's draw
    rng = np.random.default_rng(2)
    for e in np.nonzero((status & (DONE | INVALID)) == 0)[0][:40]:
        for ag in range(4):
            if S["agents"]["dead"][e, ag]:
                continue
            d = int(rng.integers(0, 5))
            assert b.policy_act(int(e), ag, d) == team_orc.simple_act(S[e:e + 1], ag, A[e, ag:ag + 1], d), (e, ag)
    assert b.policy_download().tobytes() == A.tobytes()
    b.free(dev)
    b.close()


@pytest.mark.gpu
def test_team_expand_step_and_cross_mode_refusal(pb, team_orc):
    src = pb.Batch(512, n_templates=64, teams=True)
    src.rollout(40, 21, 0, pb.ROLL_NO_RESET)
    R, rst = src.download()
    roots = np.nonzero((rst & (DONE | INVALID)) == 0)[0][:6].astype(np.uint32)
    dst = pb.Batch(6 * 1296, n_templates=1, empty=True, teams=True)
    dst.expand_step_from(src, roots, 1296, 0)
    G, gst = dst.download()
    E, est = np.repeat(R[roots], 1296), np.repeat(rst[roots], 1296)
    j = np.tile(np.arange(1296), roots.shape[0])
    mv = np.stack([j % 6, (j // 6) % 6, (j // 36) % 6, (j // 216) % 6], axis=1).astype(np.uint8)
    team_orc.env_step_batch(E, est, np.ascontiguousarray(mv))
    assert team_orc.diff_batch(G, E)[0] == -1 and (gst == est).all()
    dst.clone_from(src, roots[::-1].copy())
    # a status byte's winner field means different things in the two modes: no copies across them
    ffa = pb.Batch(6 * 1296, n_templates=1, empty=True)
    L = pb.lib()
    idx = np.ascontiguousarray(roots)
    ptr = idx.ctypes.data_as(C.c_void_p)
    assert L.pom_batch_clone(ffa.h, 0, src.h, ptr, 6) == -1 and b"team" in L.pom_last_error()
    assert L.pom_batch_expand_step(ffa.h, src.h, ptr, 6, 1296, 0) == -1 and b"team" in L.pom_last_error()
    assert L.pom_batch_clone(src.h, 0, ffa.h, ptr, 6) == -1
    assert L.pom_batch_expand_step(dst.h, ffa.h, ptr, 6, 1296, 0) == -1
    for x in (src, dst, ffa):
        x.close()


@pytest.mark.gpu
def test_team_step_overlap_matches_oracle(pb, team_orc):
    """POM_STEP_OVERLAP at 2^18 + 1500 envs (the two halves run on the tile kernel)"""
    from test_gpu_parity import _oracle_rollout
    n, ticks, seed = (1 << 18) + 1500, 30, 13
    b = pb.Batch(n, n_templates=32, max_ticks=0, teams=True)
    T, _ = b.templates()
    S, _ = b.download()
    moves_dev = b.alloc(4 * n * ticks)
    for t in range(ticks):
        b.generate_moves(moves_dev.value + 4 * n * t, seed, t, 6)
    for t in range(ticks):
        b.step(moves_dev.value + 4 * n * t, pb.STEP_AUTORESET | pb.STEP_COUNT | pb.STEP_OVERLAP)
    G, gst = b.download()
    status, stats = _oracle_rollout(team_orc, S, T, 0, ticks, seed, 6, 0)
    assert team_orc.diff_batch(G, S)[0] == -1 and (gst == status).all()
    _check_stats(b, stats)
    b.free(moves_dev)
    b.close()


@pytest.mark.gpu
def test_team_handle_ignores_geometry_switches(pb, team_orc, monkeypatch):
    """POM_TPB / POM_WS_NW pick other kernel geometries for free-for-all handles; a team handle keeps the default one"""
    from test_gpu_parity import _oracle_rollout
    monkeypatch.setenv("POM_TPB", "64")
    monkeypatch.setenv("POM_WS_NW", "16")
    b = pb.Batch(3000, n_templates=32, teams=True)
    monkeypatch.delenv("POM_TPB")
    monkeypatch.delenv("POM_WS_NW")
    T, _ = b.templates()
    S, _ = b.download()
    dev = b.alloc(4 * 3000)
    for t in range(60):
        b.generate_moves(dev, 5, t, 6)
        b.step(dev, pb.STEP_AUTORESET | pb.STEP_COUNT)
    b.rollout(40, 5, 60, 0)
    status, stats = _oracle_rollout(team_orc, S, T, 0, 100, 5, 6, 0)
    G, gst = b.download()
    assert team_orc.diff_batch(G, S)[0] == -1 and (gst == status).all()
    _check_stats(b, stats)
    b.free(dev)
    b.close()


@pytest.mark.gpu
def test_team_and_ffa_handles_couple_on_device(pb):
    """the coupling property of test_team_game_couples_with_free_for_all on two device handles driven with the same moves"""
    n, ticks = 2048, 300
    f = pb.Batch(n, n_templates=256)
    t_ = pb.Batch(n, n_templates=256, teams=True)
    mv = [f.alloc(4 * n), t_.alloc(4 * n)]

    def step(b, m):
        def run(t):
            b.generate_moves(m, 99, t, 6)
            b.step(m, 0)
            return b.download()
        return run
    earlier, wins, draws = _coupling(ticks, step(f, mv[0]), step(t_, mv[1]))
    assert earlier > 20 and wins > 20, (earlier, wins, draws)
    f.free(mv[0]); t_.free(mv[1])
    f.close(); t_.close()


BATCH_ENV_CPP = r"""
#include <cstdio>
#include <vector>
#include "pom_bboard.hpp"
using namespace bboard;
int main()
{
    const size_t n = 4096;
    BatchEnvironment team(n, 0, 0, 64, 0x1337, 0, true), ffa(n, 0, 0, 64, 0x1337, 0);
    if(!team.IsTeamGame() || ffa.IsTeamGame() || pom_batch_teams(team.Handle()) != 1 || pom_batch_teams(ffa.Handle()) != 0) return 1;
    std::vector<Move> mv(4 * n);
    for(uint32_t t = 0; t < 300; t++)
    {
        for(size_t e = 0; e < n; e++)
        {
            const uint32_t m = pom_rng_moves(5, e, t, 6);
            for(int a = 0; a < 4; a++) mv[4 * e + a] = Move((m >> (8 * a)) & 0xFF);
        }
        team.Step(mv.data());
        ffa.Step(mv.data());
    }
    long won[2] = {0, 0}, draws = 0;
    for(size_t i = 0; i < n; i++)
    {
        const uint8_t st = team.Status()[i];
        const int w = team.GetWinningTeam(i);
        if(team.GetWinner(i) != -1 || ffa.GetWinningTeam(i) != -1) return 2;
        if(!team.IsDone(i) || team.IsDraw(i) || (st & POM_STATUS_INVALID)) { if(w != -1) return 3; draws += team.IsDraw(i); continue; }
        if(w != ((st & POM_STATUS_WINNER_MASK) >> POM_STATUS_WINNER_SHIFT) || w < 0 || w > 1) return 4;
        won[w]++;
    }
    std::printf("ok %ld %ld %ld\n", won[0], won[1], draws);
    return 0;
}
"""


@pytest.mark.gpu
def test_batch_environment_team_game(pb, tmp_path):
    """bboard::BatchEnvironment(..., teams = true): IsTeamGame, GetWinningTeam (GetWinner is -1 in a team game)"""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, exe = tmp_path / "team_env.cpp", tmp_path / "team_env"
    src.write_text(BATCH_ENV_CPP)
    lib = os.path.join(root, "pomcpp_b200")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-I", os.path.join(root, "include"), "-o", str(exe), str(src),
                          os.path.join(lib, "host", "libpom_host.a"), "-L" + lib, "-lpom_b200", "-Wl,-rpath," + lib],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    _, w0, w1, _ = run.stdout.split()
    assert int(w0) > 0 and int(w1) > 0
