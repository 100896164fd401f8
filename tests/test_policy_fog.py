"""The device SimpleAgent under fog of war (pom_batch_set_policy_view).  With view v >= 0 the move of agent a is
    SimpleAgent::act( N_a( fog_state(state, a, v) ) )
fog_state = the oracle's pom_oracle_fog (the fogged State of pom_batch_observe); N_a = what SimpleActOnDevice does to a
fogged State: every other agent with x < 0 (hidden or dead) becomes dead at (0, 0).  The agent is the restatement's,
team-aware on a team handle; its draw and its memory are those of the full-state agent.  FogPolicyRestatement states
that definition on the oracle, one agent at a time, and pins the device code to it:
  CPU  the FOG instantiation of the policy built for the host (tests/fogsim) == the definition, move for move and memory
       for memory, on games, stress games and inconsistent states, views 0..16, free-for-all and team; properties (a
       large view is the full-state agent; nothing outside an agent's window changes its move); explicit cases.
  GPU  every entry point that runs the device SimpleAgent on a fogged handle == the definition."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from test_teams import TeamRestatement, TeamSim, OracleRun, _games

DONE, DRAW, INVALID, TRUNC = 0x01, 0x02, 0x10, 0x20
VIEWS = [0, 1, 2, 4, 10, 16]
MASKS = [15, 0b0110, 0b0001]


class FogPolicyRestatement:
    """The game of `orc` (free-for-all, or TeamRestatement's team game) whose SimpleAgents act on
    N_a(fog_state(state, a, view)); view < 0 = the full state.  Everything but the agent is the game's."""

    def __init__(self, orc, view, teams=False):
        self.ffa = orc
        self.game = TeamRestatement(orc) if teams else orc
        self.view = view

    def __getattr__(self, name):
        return getattr(self.game, name)

    def seen_by(self, S, a):
        """N_a(fog_state(S, a, view)) for every State of S (a copy)"""
        V = self.ffa.fog_batch(S.copy(), a, self.view)
        ag = V["agents"]
        hidden = ag["x"] < 0
        hidden[:, a] = False
        ag["dead"][hidden] = 1
        ag["x"][hidden] = 0
        ag["y"][hidden] = 0
        return V

    def simple_moves_batch(self, S, status, A, seed, env0, tick, agent_mask, moves):
        if self.view < 0:
            return self.game.simple_moves_batch(S, status, A, seed, env0, tick, agent_mask, moves)
        for a in range(4):
            if (agent_mask >> a) & 1:
                self.game.simple_moves_batch(self.seen_by(S, a), status, A, seed, env0, tick, 1 << a, moves)

    def simple_act(self, s, agent_id, st, draw):
        if self.view < 0:
            return self.game.simple_act(s, agent_id, st, draw)
        return self.game.simple_act(self.seen_by(s, agent_id), agent_id, st, draw)


class FogSim:
    """tests/fogsim: the FOG instantiation of the device SimpleAgent built for the host; records packed by tests/hostsim.
    view < 0 runs the full-state agent of tests/hostsim (free-for-all) and tests/teamsim (team)."""

    def __init__(self, so, teamsim):
        from hostsim import HostSim
        self.h = HostSim()
        self.team = teamsim
        L = self.lib = C.CDLL(so)
        vp = C.c_void_p
        L.fogsim_simple_moves.argtypes = [vp, C.c_long, vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, vp]
        L.fogsim_simple_act.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int]

    def pack(self, S, status=None):
        return self.h.pack(S, status)

    def simple_moves(self, recs, A, seed, env0, tick, mask, view, teams, moves):
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        if view >= 0:
            self.lib.fogsim_simple_moves(p(recs), recs.shape[0], p(A), seed, env0, tick, mask, view, int(teams), p(moves))
        elif teams:
            self.team.simple_moves(recs, A, seed, env0, tick, mask, moves)
        else:
            self.h.simple_moves(recs, A, seed, env0, tick, mask, moves)

    def simple_act(self, rec, agent, mem, draw, view, teams):
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        return self.lib.fogsim_simple_act(p(rec), agent, p(mem), draw, view, int(teams))


def _build(tmp_path_factory, name, src):
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    so = str(tmp_path_factory.mktemp(name) / ("lib%s.so" % name))
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-I", os.path.join(root, "include"),
                          "-I", os.path.join(root, "pomcpp_b200", "csrc"), "-o", so, os.path.join(here, src)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return so


@pytest.fixture(scope="module")
def fs(tmp_path_factory):
    return FogSim(_build(tmp_path_factory, "fogsim", "fogsim/fogsim.cpp"),
                  TeamSim(_build(tmp_path_factory, "teamsim", "teamsim/teamsim.cpp")))


def _mem_with_history(n=1):
    """agent memories holding four distinct recent positions: no _HasRPLoop, so a hunt walks towards its target"""
    mem = np.zeros((n, 4), dtype=oracle.SIMPLE_DT)
    mem["recent"][:, :] = [0x11, 0x12, 0x13, 0x14]
    mem["rp_count"][:, :] = 4
    return mem


def _drive(orc, fs, S, view, teams, mask, ticks, seed, full=None):
    """games driven by the definition's moves, auto-reset to their first state; the host build acts on the same state
    every tick.  Returns (acts compared, acts where the fogged agent differs from the full-state agent)."""
    D = FogPolicyRestatement(orc, view, teams)
    n = S.shape[0]
    S0, st = S.copy(), np.zeros(n, np.uint8)
    A = orc.simple_agents(n)
    B = A.copy()
    acts = differs = 0
    for t in range(ticks):
        mv = orc.rng_moves(seed, 0, n, t, 6)
        want, got = mv.copy(), mv.copy()
        if full is not None:
            F = mv.copy()
            FogPolicyRestatement(orc, -1, teams).simple_moves_batch(S, st, A.copy(), seed, 0, t, mask, F)
        D.simple_moves_batch(S, st, A, seed, 0, t, mask, want)
        recs, bad = fs.pack(S, st)
        assert not bad.any()
        fs.simple_moves(recs, B, seed, 0, t, mask, view, teams, got)
        assert (want == got).all(), "tick %d env %d" % (t, np.nonzero((want != got).any(1))[0][0])
        assert A.tobytes() == B.tobytes(), "memories after tick %d" % t
        alive = (S["agents"]["dead"] == 0)[:, [a for a in range(4) if (mask >> a) & 1]]
        acts += int(alive.sum())
        if full is not None:
            differs += int((F != want).any(1).sum())
        D.env_step_batch(S, st, want)
        idx = np.nonzero(st & (DONE | INVALID))[0]
        S[idx], st[idx], A[idx], B[idx] = S0[idx], 0, 0, 0
    return acts, differs


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("view", VIEWS)
def test_fogsim_games_match_definition(orc, fs, view, teams, mask):
    """games from InitState over 300 ticks with auto-reset: moves and memories, act after act"""
    S = _games(orc, 160)
    acts, differs = _drive(orc, fs, S, view, teams, mask, 300, 40 + view, full=True)
    assert acts > 160 * 300 // 2
    if view <= 4:
        assert differs > 50, differs                           # the fog does change what the agents do
    if view >= 10:
        assert differs == 0                                    # a window over the whole board is the full state


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("view", [0, 1, 2, 4, 16])
def test_fogsim_stress_games_match_definition(orc, fs, view, teams):
    """the stress regime: kicks, several bombs, long flames"""
    S = _games(orc, 160, stress=True, seed=view + 3)
    _drive(orc, fs, S, view, teams, 15, 250, 70 + view)


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("view", VIEWS)
def test_fogsim_inconsistent_states_match_definition(orc, fs, view, teams):
    """uploaded states no game reaches (tests/test_fuzz_states.py), a few ticks each"""
    from test_fuzz_states import mutated_states
    S = mutated_states(orc, 600 + view, 2000)
    recs, bad = fs.pack(S, np.zeros(S.shape[0], np.uint8))
    S = S[bad == 0].copy()
    assert S.shape[0] > 1000
    D = FogPolicyRestatement(orc, view, teams)
    n = S.shape[0]
    st = np.zeros(n, np.uint8)
    A = orc.simple_agents(n)
    B = A.copy()
    for t in range(8):
        for mask in MASKS:
            mv = orc.rng_moves(9, 0, n, 3 * t + mask, 6)
            want, got = mv.copy(), mv.copy()
            recs, bad = fs.pack(S, st)
            act = np.where(bad != 0, st | INVALID, st).astype(np.uint8)   # a state the record cannot carry does not act
            D.simple_moves_batch(S, act, A, 9, 0, 3 * t + mask, mask, want)
            fs.simple_moves(recs, B, 9, 0, 3 * t + mask, mask, view, teams, got)
            live = (act & (DONE | INVALID)) == 0
            assert (want[live] == got[live]).all(), "tick %d mask %d" % (t, mask)
            assert A.tobytes() == B.tobytes()
        D.env_step_batch(S, st, want)


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("states", ["games", "inconsistent"])
def test_large_view_is_the_full_state_agent(orc, fs, states, teams):
    """view >= 10 on game states and view 16 on every state: the moves and memories of the unfogged device policy"""
    from test_fuzz_states import mutated_states
    S = _games(orc, 400, stress=True, seed=5) if states == "games" else mutated_states(orc, 77, 2500)
    st = np.zeros(S.shape[0], np.uint8)
    if states == "games":
        for t in range(80):
            FogPolicyRestatement(orc, -1, teams).env_step_batch(S, st, orc.rng_moves(31, 0, S.shape[0], t, 6))
    recs, bad = fs.pack(S, st)
    keep = (bad == 0) & ((st & (DONE | INVALID)) == 0)
    recs = recs[keep].copy()
    n = recs.shape[0]
    A0 = orc.simple_agents(n)
    A0["recent"] = np.random.default_rng(1).integers(0, 121, A0["recent"].shape)
    A0["rp_count"] = np.random.default_rng(2).integers(0, 5, A0["rp_count"].shape)
    for t in range(4):
        full, Af = orc.rng_moves(3, 0, n, t, 6), A0.copy()
        fs.simple_moves(recs, Af, 3, 0, t, 15, -1, teams, full)
        for view in ([10, 12, 15, 16] if states == "games" else [15, 16]):
            got, Ag = orc.rng_moves(3, 0, n, t, 6), A0.copy()
            fs.simple_moves(recs, Ag, 3, 0, t, 15, view, teams, got)
            assert (got == full).all() and Ag.tobytes() == Af.tobytes(), (view, t)


def _outside_changes(S, a, view, rng):
    """S with random changes outside agent a's window: cells, bombs (added, or moved or retimed), other agents"""
    T = S.copy()
    n = T.shape[0]
    for e in range(n):
        ax, ay = int(T["agents"]["x"][e, a]), int(T["agents"]["y"][e, a])
        out = [(x, y) for y in range(11) for x in range(11) if max(abs(x - ax), abs(y - ay)) > view]
        if not out:
            continue
        for _ in range(int(rng.integers(1, 8))):
            x, y = out[int(rng.integers(0, len(out)))]
            k = int(rng.integers(0, 4))
            if k == 0:
                T["board"][e, y, x] = int(rng.choice([0, 1, 3, 6, 7, 8, (2 << 8) + int(rng.integers(0, 5))]))
            elif k == 1 and T["bombs_count"][e] < 18:
                sl = (int(T["bombs_index"][e]) + int(T["bombs_count"][e])) % 20
                T["bombs"][e, sl] = (x | (y << 4) | (int(rng.integers(0, 4)) << 8) | (int(rng.integers(1, 6)) << 12) |
                                     (int(rng.integers(1, 11)) << 16))
                T["bombs_count"][e] += 1
            elif k == 2:
                for j in range(int(T["bombs_count"][e])):
                    sl = (int(T["bombs_index"][e]) + j) % 20
                    b = int(T["bombs"][e, sl])
                    if max(abs((b & 15) - ax), abs(((b >> 4) & 15) - ay)) > view:
                        T["bombs"][e, sl] = (b & ~0xF00FF) | x | (y << 4) | (int(rng.integers(1, 11)) << 16)
            else:
                i = int(rng.integers(0, 4))
                gx, gy = int(T["agents"]["x"][e, i]), int(T["agents"]["y"][e, i])
                if i != a and max(abs(gx - ax), abs(gy - ay)) > view:
                    T["agents"]["x"][e, i], T["agents"]["y"][e, i] = x, y
                    T["agents"]["dead"][e, i] = int(rng.integers(0, 2))
    return T


@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("view", [0, 1, 2, 4, 6])
def test_nothing_outside_the_window_changes_the_move(orc, fs, view, teams):
    """cells, bombs and other agents outside agent a's window never change a's move or memory"""
    rng = np.random.default_rng(view + 10 * teams)
    S = _games(orc, 600, stress=True, seed=view)
    st = np.zeros(S.shape[0], np.uint8)
    for t in range(25):
        FogPolicyRestatement(orc, -1, teams).env_step_batch(S, st, orc.rng_moves(7, 0, S.shape[0], t, 6))
    S = S[(st & (DONE | INVALID)) == 0].copy()
    n = S.shape[0]
    for a in range(4):
        T = _outside_changes(S, a, view, rng)
        rs, bs = fs.pack(S)
        rt, bt = fs.pack(T)
        ok = (bs == 0) & (bt == 0) & (S["agents"]["dead"][:, a] == 0)
        assert ok.sum() > n // 3
        changed = int((rs[ok] != rt[ok]).any(1).sum())
        assert changed > ok.sum() // 2
        for t in range(6):
            A0 = _mem_with_history(int(ok.sum()))
            A1 = A0.copy()
            m0 = orc.rng_moves(5, 0, int(ok.sum()), t, 6)
            m1 = m0.copy()
            fs.simple_moves(rs[ok].copy(), A0, 5, 0, t, 1 << a, view, teams, m0)
            fs.simple_moves(rt[ok].copy(), A1, 5, 0, t, 1 << a, view, teams, m1)
            assert (m0[:, a] == m1[:, a]).all() and A0.tobytes() == A1.tobytes(), (a, t)


def _board(orc, agents, dead=()):
    """open board; agents = {id: (x, y)}; the others and `dead` killed"""
    S = orc.zero_state()
    for i, (x, y) in agents.items():
        orc.put_agent(S, x, y, i)
    for i in range(4):
        if i not in agents or i in dead:
            orc.kill(S, i)
    return S


def _moves(orc, fs, S, view, agent=0, teams=False, draws=range(5)):
    """{draw: (definition's move, host build's move)} for one agent with a hunt-ready memory"""
    D = FogPolicyRestatement(orc, view, teams)
    recs, bad = fs.pack(S)
    assert not bad.any()
    out = {}
    for d in draws:
        m1, m2 = _mem_with_history()[0, agent:agent + 1], _mem_with_history()[0, agent:agent + 1]
        want = D.simple_act(S, agent, m1, d)
        if view >= 0:
            assert fs.simple_act(recs[0], agent, m2, d, view, teams) == want and m1.tobytes() == m2.tobytes(), (view, d)
        out[d] = want
    return out


def test_enemy_outside_the_window_is_not_hunted(orc, fs):
    """an enemy at Manhattan distance <= 7 but outside the window is not walked towards"""
    S = _board(orc, {0: (5, 1), 1: (5, 6)})                   # Manhattan 5, Chebyshev 5
    assert set(_moves(orc, fs, S, -1).values()) == {2}        # full state: walk DOWN towards it
    for view in (1, 2, 4):
        assert len(set(_moves(orc, fs, S, view).values())) > 1, view    # random safe steps
    assert set(_moves(orc, fs, S, 0).values()) == {0}         # sees nothing: IDLE
    assert set(_moves(orc, fs, S, 5).values()) == {2}


def test_view_zero_does_not_bomb_a_neighbour(orc, fs):
    S = _board(orc, {0: (5, 5), 1: (6, 5)})
    assert set(_moves(orc, fs, S, -1).values()) == {5}
    assert 5 not in _moves(orc, fs, S, 0).values()
    assert set(_moves(orc, fs, S, 1).values()) == {5}


def test_bomb_outside_the_window_does_not_scare(orc, fs):
    """a bomb just outside the window whose blast covers the agent: the agent does not flee"""
    S = _board(orc, {0: (5, 5), 1: (0, 10)})
    S["agents"]["bombStrength"][0, 1] = 4
    orc.plant_bomb(S, 8, 5, 1, True, 1)                       # Chebyshev distance 3, about to blow up along row 5
    assert orc.is_in_danger(S, 5, 5) == 1
    calm = _board(orc, {0: (5, 5), 1: (0, 10)})
    full, fog, quiet = _moves(orc, fs, S, -1), _moves(orc, fs, S, 2), _moves(orc, fs, calm, 2)
    assert set(full.values()) == {1, 2}                       # full state: off the row, UP or DOWN
    assert fog == quiet and set(fog.values()) == {3, 4}       # fogged: the calm board's random steps
    assert _moves(orc, fs, S, 3) == full                      # in sight: it flees


def test_hunts_the_visible_enemy(orc, fs):
    """one enemy hidden, one visible, both within 7: the visible one is the target"""
    S = _board(orc, {0: (5, 5), 1: (5, 9), 3: (7, 5)})         # 1 first in order, Chebyshev 4; 3 at Chebyshev 2
    assert set(_moves(orc, fs, S, -1).values()) == {2}        # full state: DOWN towards agent 1
    assert set(_moves(orc, fs, S, 2).values()) == {4}         # fogged: RIGHT towards agent 3
    assert set(_moves(orc, fs, S, 2, teams=True).values()) == {4}    # 1 and 3 are agent 0's enemies in the team game too
    assert set(_moves(orc, fs, S, 4).values()) == {2}


def test_view_zero_plays_idle_on_game_states(orc, fs):
    """at view 0 an agent sees no walkable neighbour, no enemy and no wood: its own cell shows the agent"""
    for teams in (False, True):
        S = _games(orc, 300, stress=True, seed=9)
        st = np.zeros(300, np.uint8)
        A = orc.simple_agents(300)
        for t in range(200):
            mv = orc.rng_moves(12, 0, 300, t, 6)
            got = mv.copy()
            recs, _ = fs.pack(S, st)
            fs.simple_moves(recs, A, 12, 0, t, 15, 0, teams, got)
            live = (st & (DONE | INVALID)) == 0
            alive = S["agents"]["dead"] == 0
            assert (got[live][alive[live]] == 0).all(), t
            FogPolicyRestatement(orc, 0, teams).env_step_batch(S, st, mv)


# ----------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


@pytest.mark.gpu
def test_policy_view_setting_and_errors(pb):
    b = pb.Batch(64, n_templates=4)
    assert b.policy_view() == -1
    for v in (4, 0, 16, 1000, -1, -7):
        b.set_policy_view(v)
        assert b.policy_view() == v
    L = pb.lib()
    out = C.c_int(5)
    assert L.pom_batch_set_policy_view(None, 3) == -1
    assert L.pom_batch_get_policy_view(None, C.byref(out)) == -1 and out.value == 5
    assert L.pom_batch_get_policy_view(b.h, None) == -1
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
def test_policy_moves_match_definition(pb, orc, teams):
    """pom_batch_policy_moves (device buffer) and _host on a fogged handle, per-tick loop with auto-reset, the view and
    the agent mask changing from tick to tick; downloaded memories"""
    n, ticks, seed, env0 = 2500, 120, 21, 300
    b = pb.Batch(n, env_offset=env0, n_templates=48, max_ticks=70, teams=teams)
    T, _ = b.templates()
    S, _ = b.download()
    game = TeamRestatement(orc) if teams else orc
    R = OracleRun(game, S, T, env0, 70)
    A = orc.simple_agents(n)
    dev = b.alloc(4 * n)
    out = np.zeros(n, np.uint8)
    for t in range(ticks):
        view, mask = [4, 0, 2, 7, 16][(t // 10) % 5], MASKS[t % 3]
        b.set_policy_view(view)
        mv = orc.rng_moves(seed, env0, n, t, 6)
        want = mv.copy()
        live = (R.status & (DONE | INVALID)) == 0
        FogPolicyRestatement(orc, view, teams).simple_moves_batch(S, R.status, A, seed, env0, t, mask, want)
        if t % 2:
            got = mv.copy()
            b.policy_moves_host(got, seed, t, mask)
        else:
            pb.lib().pom_device_copy(0, dev, mv.ctypes.data_as(C.c_void_p), 4 * n)
            b.policy_moves(dev, seed, t, mask)
            b.sync()
            got = np.zeros((n, 4), np.uint8)
            pb.lib().pom_device_copy(0, got.ctypes.data_as(C.c_void_p), dev, 4 * n)
        assert (got[live] == want[live]).all(), "tick %d env %d" % (t, np.nonzero((got != want).any(1) & live)[0][0])
        b.step_host(want, out, pb.STEP_AUTORESET | pb.STEP_COUNT)
        ep = R.episode.copy()
        end = R.tick(want)
        A[R.episode != ep] = 0                                # a new episode starts with new agents
        assert (out == end).all(), "tick %d" % t
        if t % 20 == 19:
            assert b.policy_download().tobytes() == A.tobytes(), "memories, tick %d" % t
    G, gst = b.download()
    assert orc.diff_batch(G, S)[0] == -1 and (gst == R.status).all()
    assert (b.stats().as_array() == R.stats).all()
    b.free(dev)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
@pytest.mark.parametrize("view,mask", [(4, 15), (1, 0b0110), (0, 0b0001)])
def test_fused_rollout_matches_definition(pb, orc, teams, view, mask):
    """the fused kernel (small batch) with fogged SimpleAgents, with and without auto-reset: states, status bytes,
    counters, memories"""
    from test_gpu_policy import _oracle_policy_rollout
    n, ticks, seed, env0 = 1024 + 33, 160, 808, 5000
    for no_reset in (True, False):
        b = pb.Batch(n, env_offset=env0, n_templates=40, max_ticks=0 if no_reset else 90, teams=teams)
        b.set_policy_view(view)
        T, _ = b.templates()
        S, _ = b.download()
        A = orc.simple_agents(n)
        flags = pb.ROLL_SIMPLE(mask) | (pb.ROLL_NO_RESET if no_reset else 0)
        b.rollout(100, seed, 0, flags)
        b.rollout(ticks - 100, seed, 100, flags)
        G, gst = b.download()
        D = FogPolicyRestatement(orc, view, teams)
        status, stats = _oracle_policy_rollout(D, S, T, A, env0, ticks, seed, 6, 0 if no_reset else 90, mask,
                                               no_reset=no_reset)
        e, why = orc.diff_batch(G, S)
        assert e == -1, "env %d field group %d" % (e, why)
        assert (gst == status).all()
        assert (b.stats().as_array() == stats).all()
        assert b.policy_download().tobytes() == A.tobytes()
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
def test_tick_by_tick_rollout_matches_fused_and_definition(pb, orc, teams, monkeypatch):
    """>= 65536 envs run k_policy_moves + the step kernel tick by tick; bit-identical to the fused kernel
    (POM_ROLL_POLICY=fused) and, on a slice replayed by the restatement, to the definition"""
    from test_gpu_policy import _oracle_policy_rollout
    n, ticks, seed, view, mask = (1 << 16) + 4099, 45, 77, 3, 0b1011
    monkeypatch.setenv("POM_ROLL_POLICY", "fused")
    a = pb.Batch(n, n_templates=128, max_ticks=60, teams=teams)
    monkeypatch.delenv("POM_ROLL_POLICY")
    c = pb.Batch(n, n_templates=128, max_ticks=60, teams=teams)
    T, _ = c.templates()
    for x in (a, c):
        x.set_policy_view(view)
        l0 = x.launch_count()
        x.rollout(ticks, seed, 0, pb.ROLL_SIMPLE(mask))
        x.launches = x.launch_count() - l0
    assert a.launches == 1 and c.launches == 2 * ticks
    Sa, sa = a.download()
    Sc, sc = c.download()
    assert Sa.tobytes() == Sc.tobytes() and (sa == sc).all()
    assert a.stats().as_dict() == c.stats().as_dict()
    assert a.policy_download().tobytes() == c.policy_download().tobytes()
    lo, cnt = 40_001, 256
    S = np.stack([T[(lo + e) % 128] for e in range(cnt)]).astype(oracle.STATE_DT)
    M = orc.simple_agents(cnt)
    status, _ = _oracle_policy_rollout(FogPolicyRestatement(orc, view, teams), S, T, M, lo, ticks, seed, 6, 60, mask)
    assert orc.diff_batch(Sc[lo:lo + cnt], S)[0] == -1 and (sc[lo:lo + cnt] == status).all()
    assert c.policy_download(lo, cnt).tobytes() == M.tobytes()
    a.close(); c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
def test_policy_act_and_switching(pb, orc, teams):
    """pom_batch_policy_act on a fogged handle == the definition; a new view takes effect at the next call; view -1 gives
    the full-state agent's moves exactly"""
    n = 1000
    b = pb.Batch(n, n_templates=48, teams=teams)
    b.rollout(30, 3, 0, pb.ROLL_NO_RESET)
    S, status = b.download()
    A = orc.simple_agents(n)
    rng = np.random.default_rng(2)
    envs = np.nonzero((status & (DONE | INVALID)) == 0)[0][:60]
    assert envs.shape[0] >= 40
    for k, view in enumerate([4, -1, 0, 2, -1, 16]):
        b.set_policy_view(view)
        D = FogPolicyRestatement(orc, view, teams)
        for e in envs:
            for ag in range(4):
                if S["agents"]["dead"][e, ag]:
                    continue
                d = int(rng.integers(0, 5))
                assert b.policy_act(int(e), ag, d) == D.simple_act(S[e:e + 1], ag, A[e, ag:ag + 1], d), (view, e, ag)
        assert b.policy_download().tobytes() == A.tobytes(), view
    # the full-state agent through policy_moves after a fogged call: today's moves
    b.set_policy_view(-1)
    mv = orc.rng_moves(5, 0, n, 0, 6)
    want, got = mv.copy(), mv.copy()
    (TeamRestatement(orc) if teams else orc).simple_moves_batch(S, status, A, 5, 0, 0, 15, want)
    b.policy_moves_host(got, 5, 0, 15)
    live = (status & (DONE | INVALID)) == 0
    assert (got[live] == want[live]).all() and b.policy_download().tobytes() == A.tobytes()
    b.close()


BATCH_ENV_CPP = r"""
#include <cstdio>
#include <cstring>
#include <vector>
#include "pom_bboard.hpp"
using namespace bboard;
int main()
{
    const size_t n = 4096;
    BatchEnvironment env(n, 0, 0, 64, 0x1337, 0, TEAMS), raw(n, 0, 0, 64, 0x1337, 0, TEAMS);
    env.SetSimpleViewRange(4);
    if(pom_batch_set_policy_view(raw.Handle(), 4) != POM_OK) return 1;
    std::vector<Move> mv(4 * n);
    std::vector<uint8_t> m8(4 * n), st(n);
    long differ = 0;
    for(uint32_t t = 0; t < 200; t++)
    {
        for(size_t e = 0; e < n; e++)
        {
            const uint32_t m = pom_rng_moves(5, e, t, 6);
            for(int a = 0; a < 4; a++) { mv[4 * e + a] = Move((m >> (8 * a)) & 0xFF); m8[4 * e + a] = uint8_t((m >> (8 * a)) & 0xFF); }
        }
        env.Step(mv.data(), 0b0111u, 99);
        if(pom_batch_policy_moves_host(raw.Handle(), m8.data(), 99, t, 0b0111u) != POM_OK) return 2;
        if(pom_batch_step_host(raw.Handle(), m8.data(), st.data(), 0) != POM_OK) return 3;
    }
    const std::vector<State> a = env.States(), b = raw.States();
    for(size_t i = 0; i < n; i++) differ += std::memcmp(&a[i], &b[i], sizeof(State)) != 0;
    if(differ) { std::printf("differ %ld\n", differ); return 4; }
    for(size_t i = 0; i < n; i++) if(env.Status()[i] != st[i]) return 5;
    std::printf("ok\n");
    return 0;
}
"""


@pytest.mark.gpu
@pytest.mark.parametrize("teams", [False, True], ids=["ffa", "team"])
def test_batch_environment_simple_view_range(pb, tmp_path, teams):
    """bboard::BatchEnvironment::SetSimpleViewRange: a game of Step(moves, simpleMask, seed) == pom_batch_policy_moves_host
    + pom_batch_step_host with the same view"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, exe = tmp_path / "fog_env.cpp", tmp_path / "fog_env"
    src.write_text(BATCH_ENV_CPP.replace("TEAMS", "true" if teams else "false"))
    lib = os.path.join(root, "pomcpp_b200")
    out = subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-I", os.path.join(root, "include"), "-o", str(exe), str(src),
                          os.path.join(lib, "host", "libpom_host.a"), "-L" + lib, "-lpom_b200", "-Wl,-rpath," + lib],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
