"""The step kernels at the edges of their integer widths and fixed capacities, where a kernel can be subtly wrong while every
ordinary-size test passes:
  A  the 16-bit timeStep ceiling: an env that would pass 65535 is aborted as INVALID (pomcore::env_post), in every entry
     point that steps, and against max_ticks (a uint32 compared with the 16-bit episode length);
  B  the 16-bit per-lane episode counters (EpisodeAcc) of fused launches that finish more than 65535 episodes per lane;
  C  global env indices past 2^32 (template index, RNG keys) and the wrap of the uint32 tick counter;
  D  the finished-env list of pom_batch_step_compact at and past the 480 entries a CTA keeps in shared memory, and its
     clipping to the caller's capacity.
The references are the restatement (oracle/) with the ceiling rule on top (ceiling_step) and a vectorised replay of the
episode rule (Replay); the one CPU test checks that replay against test_gpu_parity._oracle_rollout."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
from test_gpu_parity import _oracle_rollout
from test_gpu_policy import _oracle_policy_rollout
from test_rewards import reward_definition
from test_teams import team_orc  # noqa: F401  (fixture: the team game on the restatement)

DONE, DRAW, INVALID, TRUNC = 0x01, 0x02, 0x10, 0x20
ENDED = DONE | INVALID | TRUNC
CEIL = 65535
U32 = 0xFFFFFFFF


# ----------------------------------------------------------------------------------------------------------- references


def ceiling_step(orc, S, status, moves, flags=None):
    """orc.env_step_batch with the 16-bit timeStep of the record: a stepped env whose timeStep comes out as 65536 gets
    65535 back and status |= INVALID; its board, agents and any DONE / winner / DRAW bits of the tick stay"""
    stepped = (status & (DONE | INVALID)) == 0
    orc.env_step_batch(S, status, np.ascontiguousarray(moves), flags)
    top = stepped & (S["timeStep"] > CEIL)
    S["timeStep"][top] = CEIL
    status[top] |= INVALID


class Ceiling:
    """a restatement whose env_step_batch is ceiling_step (for the replays of other files, which take the restatement)"""

    def __init__(self, orc):
        self.o = orc

    def __getattr__(self, name):
        return getattr(self.o, name)

    def env_step_batch(self, S, status, moves, flags=None):
        ceiling_step(self.o, S, status, moves, flags)


def raw_step(orc, S, status, moves):
    """POM_STEP_RAW: bare Step on every env that is not INVALID (done ones too), no timeStep++, so no ceiling"""
    live = np.nonzero((status & INVALID) == 0)[0]
    sub = S[live]
    f = np.zeros(live.shape[0], np.uint8)
    orc.step_batch(sub, np.ascontiguousarray(moves[live]), f)
    S[live] = sub
    status[live[(f & 0x3E) != 0]] |= INVALID


class Replay:
    """Vectorised replay of the episode rule of pom_batch_rollout (and of pom_batch_step with AUTORESET): step the live
    envs on the restatement under the ceiling rule, freeze finished ones, truncate at max_ticks, count with the precedence
    DONE > TRUNCATED > aborted, reset to T[(env0 + e + episode) % nT].  env0 is a Python int below 2^63."""

    def __init__(self, orc, S, T, env0=0, max_ticks=0, no_reset=False):
        n = S.shape[0]
        self.o, self.S, self.T, self.max_ticks, self.no_reset = orc, S, T, max_ticks, no_reset
        self.idx = np.uint64(env0) + np.arange(n, dtype=np.uint64)
        self.status = np.zeros(n, np.uint8)
        self.episode = np.zeros(n, np.uint64)
        self.stats = np.zeros(10, np.int64)

    def tick(self, mv, autoreset=True):
        """one tick; returns every env's end-of-tick status byte before any reset (what status_out reports)"""
        S, st = self.S, self.status
        live = (st & ENDED) == 0
        self.stats[0] += int(live.sum())
        if live.all():
            ceiling_step(self.o, S, st, mv)
        else:
            li = np.nonzero(live)[0]
            sub, sst = S[li], st[li]
            ceiling_step(self.o, sub, sst, np.ascontiguousarray(mv[li]))
            S[li], st[li] = sub, sst
        if not autoreset:
            return st.copy()
        if self.max_ticks:
            st[live & ((st & DONE) == 0) & (S["timeStep"] >= self.max_ticks)] |= TRUNC
        end = st.copy()
        f = np.nonzero(live & ((st & ENDED) != 0))[0]
        if f.size:
            e = st[f].astype(np.int64)
            done = (e & DONE) != 0
            draw = done & ((e & DRAW) != 0)
            trunc = ~done & ((e & TRUNC) != 0)
            s = self.stats
            s[1] += f.size
            s[2:6] += np.bincount((e[done & ~draw] >> 2) & 3, minlength=4)
            s[6] += int(draw.sum())
            s[7] += int(trunc.sum())
            s[8] += int(S["timeStep"][f].astype(np.int64).sum())
            s[9] += int((~done & ~trunc).sum())
            if not self.no_reset:
                self.episode[f] += np.uint64(1)
                S[f] = self.T[((self.idx[f] + self.episode[f]) % np.uint64(self.T.shape[0])).astype(np.int64)]
                st[f] = 0
        return end


def replay(orc, S, T, env0, ticks, seed, nact, max_ticks, tick0=0, no_reset=False):
    """_oracle_rollout's interface on Replay: ticks are (tick0 + k) mod 2^32"""
    R = Replay(orc, S, T, env0, max_ticks, no_reset)
    for k in range(ticks):
        R.tick(orc.rng_moves(seed, env0, S.shape[0], (tick0 + k) & U32, nact))
    return R.status, R.stats


def _oracle_templates(orc, nT):
    T = orc.zero_state(nT)
    for k, seed in enumerate(oracle.clean_seeds(nT)):
        assert orc.init_state(T[k:k + 1], seed) == 0
    return T


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("no_reset", [False, True], ids=["reset", "no-reset"])
def test_replay_matches_oracle_rollout(orc, no_reset):
    """the vectorised replay == the loop of test_gpu_parity._oracle_rollout: resets from a pool whose index passes 2^32,
    truncation, and (no_reset) envs that stay frozen once finished"""
    n, ticks, seed, env0, nT = 203, 150, 3, 2 ** 32 - 100, 24
    T = _oracle_templates(orc, nT)
    S0 = T[(env0 + np.arange(n)) % nT].copy()
    A = S0.copy()
    st_a, stats_a = _oracle_rollout(orc, A, T, env0, ticks, seed, 6, 40, no_reset=no_reset)
    B = S0.copy()
    st_b, stats_b = replay(orc, B, T, env0, ticks, seed, 6, 40, no_reset=no_reset)
    assert orc.diff_batch(A, B)[0] == -1
    assert (st_a == st_b).all()
    assert (stats_a == stats_b).all(), (stats_a, stats_b)
    assert stats_a[7] > 0 and stats_a[1] > stats_a[7]           # truncations and game ends
    if no_reset:
        assert ((st_a & ENDED) != 0).sum() > n // 2             # most envs finished and stayed frozen
    else:
        assert stats_a[1] > n


# ----------------------------------------------------------------------------------------------------------- GPU helpers


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


def _to_dev(pb, dst, a):
    pb._ck(pb.lib().pom_device_copy(0, dst, a.ctypes.data_as(C.c_void_p), a.nbytes))


def _from_dev(pb, a, src):
    pb._ck(pb.lib().pom_device_copy(0, a.ctypes.data_as(C.c_void_p), src, a.nbytes))
    return a


def _sm_count():
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    dev, v = C.c_int(), C.c_int()
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetAttribute(C.byref(v), 16, dev) == 0      # CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT
    return v.value


_NEAR = {}


def _near_ceiling(pb, orc, n=3017, kills=True):
    """n running mid-game states (a 14-tick NO_RESET rollout: bombs, flames, powerups) at timeStep 65533 + e % 3.
    kills: env e % 8 == 5 keeps one agent alive and e % 8 == 6 none, both at 65535 (the ceiling tick ends the game too:
    DONE | INVALID with a winner, DONE | DRAW | INVALID); e % 16 == 7 has nobody alive at 65534 (DONE | DRAW first)."""
    key = (n, kills)
    if key not in _NEAR:
        src = pb.Batch(2 * n + 64, n_templates=64)
        src.rollout(14, 4141, 0, pb.ROLL_NO_RESET)
        S, st = src.download()
        src.close()
        S = np.ascontiguousarray(S[st == 0][:n])
        assert S.shape[0] == n
        e = np.arange(n)
        S["timeStep"] = CEIL - 2 + e % 3
        if kills:
            for i in np.nonzero((e % 8 == 5) | (e % 8 == 6) | (e % 16 == 7))[0]:
                alive = np.nonzero(S["agents"]["dead"][i] == 0)[0]
                orc.kill(S[i:i + 1], *[int(a) for a in (alive[1:] if i % 8 == 5 else alive)])
                S["timeStep"][i] = CEIL if i % 8 != 7 else CEIL - 1
        _NEAR[key] = S
    return _NEAR[key].copy()


def _tiled(S, n):
    return np.ascontiguousarray(S[np.arange(n) % S.shape[0]])


def _assert_ceiling_outcomes(ends):
    """the ticks saw the ceiling alone, the ceiling with a winner and the ceiling with a draw"""
    e = np.concatenate(ends)
    kind = e & (DONE | DRAW | INVALID)
    assert (kind == INVALID).any()
    assert (kind == DONE | INVALID).any()
    assert (kind == DONE | DRAW | INVALID).any()


def _same(orc, G, gst, S, st, what):
    e, why = orc.diff_batch(G, S)
    assert e == -1, "%s: env %d field group %d" % (what, e, why)
    assert (gst == st).all(), "%s: status of env %d: %#x != %#x" % (what, np.nonzero(gst != st)[0][0],
                                                                    gst[gst != st][0], st[gst != st][0])


# ----------------------------------------------------------------------------------------------------------- A: ceiling


AR, COUNT = 0x2, 0x4
PER_TICK = {"frozen": 0, "spec": AR | COUNT, "generic": AR, "raw": 0x1, "step_host": AR | COUNT,
            "step_host_pinned": AR | COUNT, "tile": AR | COUNT, "overlap": AR | COUNT | 0x8}


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PER_TICK))
def test_ceiling_per_tick_step(pb, orc, path, monkeypatch):
    """pom_batch_step (flags 0: frozen after the INVALID tick; AUTORESET | COUNT on aligned moves: the SPEC image;
    AUTORESET alone: the generic image; POM_STEP_RAW: no timeStep++, never at the ceiling), pom_batch_step_host with
    pageable and pinned buffers, POM_STEP_KERNEL=tile and POM_STEP_OVERLAP: every field of every env after every tick,
    the status bytes, and the counters (sum_episode_len + 65535 per aborted episode)"""
    flags, seed, env0, ticks = PER_TICK[path], 61, 7, 4
    S = _near_ceiling(pb, orc)
    n = (1 << 18) + 1500 if path == "overlap" else S.shape[0]
    S = _tiled(S, n)
    t0 = S["timeStep"].copy()
    if path == "tile":
        monkeypatch.setenv("POM_STEP_KERNEL", "tile")
    b = pb.Batch(n, env_offset=env0, n_templates=24, max_ticks=0, empty=True)
    monkeypatch.delenv("POM_STEP_KERNEL", raising=False)
    b.upload(S)
    T, _ = b.templates()
    R = Replay(orc, S, T, env0)
    dev = b.alloc(4 * n)
    owners = []
    if path == "step_host_pinned":
        mvp, o1 = pb.pinned_array((n, 4), np.uint8)
        out, o2 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2]
    else:
        out = np.zeros(n, np.uint8)
    ends = []
    for t in range(ticks):
        mv = orc.rng_moves(seed, env0, n, t, 6)
        if path == "step_host":
            b.step_host(mv, out, flags)
        elif path == "step_host_pinned":
            mvp[:] = mv
            b.step_host(mvp, out, flags)
        else:
            b.generate_moves(dev, seed, t, 6)
            b.step(dev, flags)
        if path == "raw":
            raw_step(orc, R.S, R.status, mv)
            end = R.status.copy()
        else:
            end = R.tick(mv, autoreset=bool(flags & AR))
        ends.append(end)
        if path.startswith("step_host"):
            assert (out == end).all(), "tick %d: status_out of env %d" % (t, np.nonzero(out != end)[0][0])
        if path != "overlap" or t == ticks - 1:
            G, gst = b.download()
            _same(orc, G, gst, R.S, R.status, "%s tick %d" % (path, t))
    got = b.stats().as_array()
    if flags & AR:
        want = R.stats.copy()
        if not flags & COUNT:
            want[0] = 0
        assert (got == want).all(), (b.stats().as_dict(), want)
        assert want[9] > 0 and want[8] >= CEIL * want[9]
    else:
        assert not got.any()
    if path == "raw":
        assert (G["timeStep"] == t0).all()                      # no timeStep++: stays at 65535, never invalidated by it
        assert (gst & INVALID).sum() < n // 100
    else:
        _assert_ceiling_outcomes(ends)
        if not flags & AR:                                      # every env ended, nearly all of them at the ceiling
            assert ((gst & (DONE | INVALID)) != 0).all() and ((gst & INVALID) != 0).mean() > 0.6
    b.free(dev)
    for o in owners:
        pb.pinned_free(o)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["spec", "harmless", "no_reset", "step_seq"])
def test_ceiling_rollout(pb, orc, kind):
    """pom_batch_rollout (the SPEC image, HARMLESS, NO_RESET) and pom_batch_step_seq across the ceiling"""
    S = _near_ceiling(pb, orc)
    n, seed, env0, ticks = S.shape[0], 62, 11, 5
    nact = 5 if kind == "harmless" else 6
    b = pb.Batch(n, env_offset=env0, n_templates=24, max_ticks=0, empty=True)
    b.upload(S)
    T, _ = b.templates()
    if kind == "step_seq":
        seq = b.alloc(4 * n * ticks)
        for t in range(ticks):
            b.generate_moves(seq.value + 4 * n * t, seed, t, 6)
        b.step_seq(seq, ticks, 0)
    else:
        b.rollout(ticks, seed, 0, {"spec": 0, "harmless": pb.ROLL_HARMLESS, "no_reset": pb.ROLL_NO_RESET}[kind])
    status, stats = replay(orc, S, T, env0, ticks, seed, nact, 0, no_reset=kind == "no_reset")
    G, gst = b.download()
    _same(orc, G, gst, S, status, kind)
    assert (b.stats().as_array() == stats).all(), (b.stats().as_dict(), stats)
    assert stats[9] > 0 and stats[2:6].sum() > 0 and stats[6] > 0
    if kind == "step_seq":
        b.free(seq)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3017, (1 << 16) + 99], ids=["fused", "tick-by-tick"])
def test_ceiling_simple_agent_rollout(pb, orc, n):
    """rollouts with four SimpleAgents across the ceiling: the fused kernel (n < 65536) and the tick-by-tick path (the
    FREEZE image of k_step_ws) against pom_batch_policy_moves + pom_batch_step on a twin handle, and the replay"""
    S = _tiled(_near_ceiling(pb, orc), n)
    seed, env0, ticks = 63, 5, 4
    a = pb.Batch(n, env_offset=env0, n_templates=24, empty=True)
    c = pb.Batch(n, env_offset=env0, n_templates=24, empty=True)
    a.upload(S)
    c.upload(S)
    l0 = a.launch_count()
    a.rollout(ticks, seed, 0, pb.ROLL_SIMPLE(15))
    assert a.launch_count() - l0 == (1 if n < (1 << 16) else 2 * ticks)
    dev = c.alloc(4 * n)
    for t in range(ticks):
        c.generate_moves(dev, seed, t, 6)
        c.policy_moves(dev, seed, t, 15)
        c.step(dev, AR | COUNT)
    A, sa = a.download()
    B, sc = c.download()
    assert A.tobytes() == B.tobytes() and (sa == sc).all()
    assert (a.stats().as_array() == c.stats().as_array()).all(), (a.stats().as_dict(), c.stats().as_dict())
    assert a.policy_download().tobytes() == c.policy_download().tobytes()
    if n < (1 << 16):
        T, _ = a.templates()
        Ag = orc.simple_agents(n)
        status, stats = _oracle_policy_rollout(Ceiling(orc), S, T, Ag, env0, ticks, seed, 6, 0, 15)
        _same(orc, A, sa, S, status, "fused vs oracle")
        assert (a.stats().as_array() == stats).all() and a.policy_download().tobytes() == Ag.tobytes()
    assert a.stats().invalid > 0
    c.free(dev)
    a.close()
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("raw", [False, True], ids=["env-step", "raw"])
def test_ceiling_expand_step(pb, orc, raw):
    """pom_batch_expand_step from roots at 65535: every child is INVALID with its own stepped state; with POM_STEP_RAW
    every child keeps timeStep 65535 and none is invalidated by the ceiling"""
    S = _near_ceiling(pb, orc)[:8].copy()
    S["timeStep"] = CEIL
    roots = np.arange(8, dtype=np.uint32)
    src = pb.Batch(8, n_templates=1, empty=True)
    src.upload(S)
    dst = pb.Batch(8 * 1296, n_templates=1, empty=True)
    dst.expand_step_from(src, roots, 1296, 0x1 if raw else 0)
    G, gst = dst.download()
    E = np.repeat(S, 1296)
    est = np.zeros(E.shape[0], np.uint8)
    j = np.tile(np.arange(1296), 8)
    mv = np.ascontiguousarray(np.stack([j % 6, (j // 6) % 6, (j // 36) % 6, (j // 216) % 6], axis=1).astype(np.uint8))
    (raw_step if raw else ceiling_step)(orc, E, est, mv)
    _same(orc, G, gst, E, est, "children")
    assert (G["timeStep"] == CEIL).all()
    if raw:
        assert (gst & INVALID).sum() < G.shape[0] // 100
    else:
        assert ((gst & INVALID) != 0).all()
        _assert_ceiling_outcomes([gst])
    src.close()
    dst.close()


@pytest.mark.gpu
@pytest.mark.parametrize("max_ticks", [65535, 65536, 70000, 800])
def test_ceiling_against_max_ticks(pb, orc, max_ticks):
    """today's definition: 65535 truncates at 65535 and never reaches the ceiling; 65536 and 70000 never truncate and
    abort at the ceiling (70000: an env uploaded at 4463 must not truncate, which catches max_ticks narrowed to 16
    bits); 800 with an env uploaded at 65535 gives INVALID | TRUNCATED, counted as truncated"""
    S = _near_ceiling(pb, orc, kills=False)
    n, seed, env0, ticks = S.shape[0], 64, 3, 3
    g = np.arange(n) % 4
    S["timeStep"] = np.array([CEIL - 2, CEIL - 1, CEIL, 4463])[g]
    b = pb.Batch(n, env_offset=env0, n_templates=24, max_ticks=max_ticks, empty=True)
    b.upload(S)
    T, _ = b.templates()
    R = Replay(orc, S, T, env0, max_ticks)
    out = np.zeros(n, np.uint8)
    ends = []
    for t in range(ticks):
        mv = orc.rng_moves(seed, env0, n, t, 6)
        b.step_host(mv, out, AR | COUNT)
        ends.append(R.tick(mv))
        assert (out == ends[-1]).all(), "tick %d env %d" % (t, np.nonzero(out != ends[-1])[0][0])
    G, gst = b.download()
    _same(orc, G, gst, R.S, R.status, "max_ticks %d" % max_ticks)
    assert (b.stats().as_array() == R.stats).all(), (b.stats().as_dict(), R.stats)
    e0 = ends[0]
    running = (e0 & DONE) == 0
    if max_ticks == 65535:
        assert ((e0[(g == 1) & running] & (TRUNC | INVALID)) == TRUNC).all()
        assert ((ends[1][(g == 0) & running & ((ends[1] & DONE) == 0)] & (TRUNC | INVALID)) == TRUNC).all()
    elif max_ticks in (65536, 70000):
        assert not any(((e & TRUNC) != 0).any() for e in ends)
        assert ((e0[g == 2] & INVALID) != 0).all()
        assert (e0[g == 3] == 0).sum() > 0.9 * (g == 3).sum()
    else:
        assert ((e0[(g == 2) & running] & (TRUNC | INVALID)) == TRUNC | INVALID).all()
        assert b.stats().truncated >= ((g == 2) & running).sum()


@pytest.mark.gpu
def test_ceiling_natural_harmless_run(pb, orc):
    """one fused HARMLESS launch of 65540 ticks from fresh templates, max_ticks = 0, 300 envs (ragged tiles): harmless
    agents never bomb, so every env reaches the ceiling on its 65536th tick, is aborted, reset and plays 4 more ticks"""
    n, ticks, seed = 300, 65540, 65
    b = pb.Batch(n, n_templates=16, max_ticks=0)
    T, _ = b.templates()
    S, _ = b.download()
    b.rollout(ticks, seed, 0, pb.ROLL_HARMLESS)
    s = b.stats()
    assert s.invalid == s.episodes == n, s.as_dict()
    assert s.sum_episode_len == CEIL * n and s.env_steps == ticks * n
    status, stats = replay(orc, S, T, 0, ticks, seed, 5, 0)
    G, gst = b.download()
    _same(orc, G, gst, S, status, "after 65540 ticks")
    assert (s.as_array() == stats).all()
    b.close()


@pytest.mark.gpu
def test_ceiling_step_compact(pb, orc):
    """pom_batch_step_compact across the ceiling: done bits and finished-env list against a twin's status bytes"""
    S = _near_ceiling(pb, orc)
    n = S.shape[0]
    a = pb.Batch(n, env_offset=9, n_templates=24, empty=True)
    c = pb.Batch(n, env_offset=9, n_templates=24, empty=True)
    a.upload(S)
    c.upload(S)
    L = _ListBuffers(pb, a, n)
    rng = np.random.default_rng(66)
    for t in range(3):
        mv = rng.integers(0, 6, (n, 4), dtype=np.uint8)
        stepped = (c.status() & (DONE | INVALID)) == 0
        want = np.zeros(n, np.uint8)
        c.step_host(mv, want, AR | COUNT)
        L.tick(pb.joint_of_moves(mv), n, AR | COUNT)
        L.check(stepped & ((want & ENDED) != 0), want)
        if t == 0:
            _assert_ceiling_outcomes([want])
    assert a.download()[0].tobytes() == c.download()[0].tobytes()
    assert (a.stats().as_array() == c.stats().as_array()).all()
    L.free()
    a.close()
    c.close()


@pytest.mark.gpu
def test_ceiling_step_rewards(pb, orc):
    """pom_batch_step_rewards: all-zero rewards for an INVALID tick, DONE | INVALID included; the counters count a
    DONE | INVALID episode as a win (DONE first), the rewards say 0.  Both are the documented definitions."""
    S = _near_ceiling(pb, orc)
    n, seed, env0 = S.shape[0], 67, 2
    b = pb.Batch(n, env_offset=env0, n_templates=24, empty=True)
    b.upload(S)
    T, _ = b.templates()
    R = Replay(orc, S, T, env0)
    dev = b.alloc(4 * n)
    rw, o1 = pb.pinned_array((n, 4), np.int8)
    st, o2 = pb.pinned_array((n,), np.uint8)
    won_invalid = 0
    for t in range(3):
        b.generate_moves(dev, seed, t, 6)
        stepped = (R.status & (DONE | INVALID)) == 0
        b.step_rewards(dev, rw, st, AR | COUNT)
        b.sync()
        end = R.tick(orc.rng_moves(seed, env0, n, t, 6))
        assert (st == end).all()
        want = reward_definition(stepped, end, R.S["agents"]["dead"] != 0, False)
        assert (rw == want).all(), "tick %d env %d" % (t, np.nonzero((rw != want).any(1))[0][0])
        assert not rw[(end & INVALID) != 0].any()
        won_invalid += int(((end & (DONE | DRAW | INVALID)) == DONE | INVALID).sum())
    assert won_invalid > 0
    s = b.stats()
    assert (s.as_array() == R.stats).all(), (s.as_dict(), R.stats)
    assert sum(s.wins) >= won_invalid
    b.free(dev)
    pb.pinned_free(o1)
    pb.pinned_free(o2)
    b.close()


@pytest.mark.gpu
def test_ceiling_step_radio(pb, team_orc):
    """pom_batch_step_radio on a radio handle: the messages of the INVALID tick are latched (a dead agent's as 0); the
    auto-reset of an ended env clears them, a running env keeps them"""
    orc = team_orc
    S = _near_ceiling(pb, orc.o)
    n, seed = S.shape[0], 68
    b = pb.Batch(n, n_templates=24, teams=True, radio=True, empty=True)
    T, _ = b.templates()
    dev = b.alloc(4 * n)
    msgs, o1 = pb.pinned_array((n, 4), np.uint8)
    st, o2 = pb.pinned_array((n,), np.uint8)
    rng = np.random.default_rng(seed)
    for flags in (0, AR | COUNT):
        b.upload(S)
        R = Replay(orc, S.copy(), T)
        for t in range(3):
            msgs[:] = rng.integers(0, 64, (n, 4), dtype=np.uint8)
            stepped = (R.status & (DONE | INVALID)) == 0
            alive = R.S["agents"]["dead"] == 0                  # a dead agent's message is silenced
            before = b.radio_download()
            b.generate_moves(dev, seed, t, 6)
            b.step_radio(dev, msgs, None, st, flags)
            b.sync()
            end = R.tick(orc.rng_moves(seed, 0, n, t, 6), autoreset=bool(flags))
            assert (st == end).all(), "tick %d" % t
            got = b.radio_download()
            reset = stepped & ((end & ENDED) != 0) if flags else np.zeros(n, bool)
            want = np.where(stepped[:, None], np.where(alive, msgs, 0), before)
            want[reset] = 0
            assert (got == want).all(), "flags %d tick %d env %d" % (flags, t, np.nonzero((got != want).any(1))[0][0])
            if flags == 0 and t == 0:
                assert ((end[stepped] & INVALID) != 0).sum() > n // 3
        G, gst = b.download()
        _same(orc, G, gst, R.S, R.status, "radio flags %d" % flags)
    b.free(dev)
    pb.pinned_free(o1)
    pb.pinned_free(o2)
    b.close()


@pytest.mark.gpu
def test_ceiling_step_observe(pb, orc):
    """pom_batch_step_observe: after the ceiling tick the planes equal the restatement's, bytes 490-491 (timeStep) read
    0xFF 0xFF"""
    S = _near_ceiling(pb, orc)
    n, seed = S.shape[0], 69
    b = pb.Batch(n, n_templates=24, empty=True)
    b.upload(S)
    T, _ = b.templates()
    R = Replay(orc, S, T)
    dev = b.alloc(4 * n)
    stride = int(pb.lib().pom_batch_obs_stride(b.h))
    obs = b.alloc(2 * stride * pb.OBS_BYTES)
    for t in range(3):
        b.generate_moves(dev, seed, t, 6)
        b.step_observe(dev, obs, 0b1001, 4, 0)
        R.tick(orc.rng_moves(seed, 0, n, t, 6), autoreset=False)
    b.sync()
    host = _from_dev(pb, np.zeros((2, stride, pb.OBS_BYTES), np.uint8), obs)[:, :n]
    for k, agent in enumerate((0, 3)):
        want = orc.observe_planes_batch(R.S, agent, 4)
        assert (host[k] == want).all(), "agent %d env %d" % (agent, np.nonzero((host[k] != want).any(1))[0][0])
    top = R.S["timeStep"] == CEIL
    assert top.mean() > 0.6 and ((R.status[top] & INVALID) != 0).mean() > 0.6
    assert (host[:, top, 490:492] == 0xFF).all()
    b.free(dev)
    b.free(obs)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["step", "rollout"])
def test_ceiling_team_handle(pb, team_orc, path):
    """the team game's episode rule at the ceiling: one team left on the ceiling tick is DONE | INVALID with the team
    as winner"""
    orc = team_orc
    S = _near_ceiling(pb, orc.o)
    n, seed, env0, ticks = S.shape[0], 70, 13, 4
    b = pb.Batch(n, env_offset=env0, n_templates=24, teams=True, empty=True)
    b.upload(S)
    T, _ = b.templates()
    R = Replay(orc, S, T, env0)
    dev = b.alloc(4 * n)
    if path == "rollout":
        b.rollout(ticks, seed, 0, 0)
    ends = []
    for t in range(ticks):
        if path == "step":
            b.generate_moves(dev, seed, t, 6)
            b.step(dev, AR | COUNT)
        ends.append(R.tick(orc.rng_moves(seed, env0, n, t, 6)))
    G, gst = b.download()
    _same(orc, G, gst, R.S, R.status, "team " + path)
    assert (b.stats().as_array() == R.stats).all(), (b.stats().as_dict(), R.stats)
    _assert_ceiling_outcomes(ends)
    b.free(dev)
    b.close()


# ----------------------------------------------------------------------------------------------------------- B: counters


def _first_tick_never_ends(orc, T):
    """no template ends or turns invalid on its first tick, under any of the 1296 joint actions"""
    j = np.tile(np.arange(1296), T.shape[0])
    mv = np.ascontiguousarray(np.stack([j % 6, (j // 6) % 6, (j // 36) % 6, (j // 216) % 6], axis=1).astype(np.uint8))
    E = np.repeat(T, 1296)
    st = np.zeros(E.shape[0], np.uint8)
    orc.env_step_batch(E, st, mv)
    assert not st.any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["spec", "harmless", "step_seq", "simple"])
def test_counters_past_16_bits(pb, orc, kind):
    """max_ticks = 1: every episode is one tick long and truncated, and one fused launch of 70000 ticks finishes more
    than 65535 episodes per lane, past the width of the per-lane counters.  The counters are exact, and every env ends
    as template (env_offset + e + 70000) % 24 with status 0."""
    ticks, off, nT = 70000, 1000003, 24
    n = 64 if kind in ("step_seq", "simple") else 4005
    b = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=1)
    T, _ = b.templates()
    _first_tick_never_ends(orc, T)
    if kind == "step_seq":
        seq = b.alloc(4 * n * ticks)
        _to_dev(pb, seq, np.random.default_rng(71).integers(0, 6, (ticks, n, 4), dtype=np.uint8))
        b.step_seq(seq, ticks, 0)
        b.sync()
        b.free(seq)
    else:
        b.rollout(ticks, 72, 0, {"spec": 0, "harmless": pb.ROLL_HARMLESS, "simple": pb.ROLL_SIMPLE(15)}[kind])
    want = np.zeros(10, np.int64)
    want[[0, 1, 7, 8]] = ticks * n
    assert (b.stats().as_array() == want).all(), b.stats().as_dict()
    G, gst = b.download()
    _same(orc, G, gst, T[(off + np.arange(n) + ticks) % nT], np.zeros(n, np.uint8), kind)
    b.close()


# ----------------------------------------------------------------------------------------------------------- C: 2^32


OFFSETS = [2 ** 32 - 1500, 2 ** 32 + 7, 2 ** 40 + 3, 2 ** 62 + 11]
offsets = pytest.mark.parametrize("off", OFFSETS, ids=hex)
pools = pytest.mark.parametrize("nT", [24, 64], ids=["pool24", "pool64"])


def _template_index(off, n, nT, episode=0):
    return ((np.uint64(off) + np.arange(n, dtype=np.uint64) + np.uint64(episode)) % np.uint64(nT)).astype(np.int64)


@pytest.mark.gpu
@offsets
@pools
def test_offsets_init_reset_and_moves(pb, orc, off, nT):
    """env e starts, and after pom_batch_reset starts again, as template (off + e) % nT; pom_batch_generate_moves draws
    the moves of global env off + e"""
    n, seed = 3000, 73
    b = pb.Batch(n, env_offset=off, n_templates=nT)
    T, _ = b.templates()
    S, st = b.download()
    assert S.tobytes() == T[_template_index(off, n, nT)].tobytes() and not st.any()
    dev = b.alloc(4 * n)
    for tick in (0, 17, U32):
        b.generate_moves(dev, seed, tick, 6)
        b.sync()
        got = _from_dev(pb, np.zeros((n, 4), np.uint8), dev)
        assert (got == orc.rng_moves(seed, off, n, tick, 6)).all(), "tick %d" % tick
        b.step(dev, AR | COUNT)
    b.reset()
    S, st = b.download()
    assert S.tobytes() == T[_template_index(off, n, nT)].tobytes() and not st.any()
    assert not b.stats().as_array().any()
    b.free(dev)
    b.close()


@pytest.mark.gpu
@offsets
@pools
@pytest.mark.parametrize("form", ["spec", "generic", "tile"])
def test_offsets_per_tick_step(pb, orc, off, nT, form, monkeypatch):
    """90 ticks with max_ticks = 60 and auto-reset: the reset's template index past 2^32 (the 64-bit % path for a pool
    of 24, the mask for 64) in the SPEC image, the generic image and the tile kernel"""
    n, ticks, seed = 3000, 90, 74
    flags = AR if form == "generic" else AR | COUNT
    if form == "tile":
        monkeypatch.setenv("POM_STEP_KERNEL", "tile")
    b = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=60)
    monkeypatch.delenv("POM_STEP_KERNEL", raising=False)
    T, _ = b.templates()
    S, _ = b.download()
    dev = b.alloc(4 * n)
    for t in range(ticks):
        b.generate_moves(dev, seed, t, 6)
        b.step(dev, flags)
    status, stats = replay(orc, S, T, off, ticks, seed, 6, 60)
    G, gst = b.download()
    _same(orc, G, gst, S, status, form)
    if form == "generic":
        stats[0] = 0
    assert (b.stats().as_array() == stats).all(), (b.stats().as_dict(), stats)
    assert stats[7] > 0 and stats[1] > n
    b.free(dev)
    b.close()


@pytest.mark.gpu
@offsets
@pools
@pytest.mark.parametrize("kind", ["spec", "harmless", "simple"])
def test_offsets_rollout(pb, orc, off, nT, kind):
    """fused rollouts (the SPEC image, HARMLESS, SimpleAgents), 150 ticks over two launches: the hoisted 64-bit RNG key
    and the reset's template index"""
    n, ticks, seed = 3000, 150, 75
    flags = {"spec": 0, "harmless": pb.ROLL_HARMLESS, "simple": pb.ROLL_SIMPLE(0b1011)}[kind]
    b = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=60)
    T, _ = b.templates()
    S, _ = b.download()
    b.rollout(100, seed, 0, flags)
    b.rollout(ticks - 100, seed, 100, flags)
    if kind == "simple":
        A = orc.simple_agents(n)
        status, stats = _oracle_policy_rollout(orc, S, T, A, off, ticks, seed, 6, 60, 0b1011)
        assert b.policy_download().tobytes() == A.tobytes()
    else:
        status, stats = replay(orc, S, T, off, ticks, seed, 5 if kind == "harmless" else 6, 60)
    G, gst = b.download()
    _same(orc, G, gst, S, status, kind)
    assert (b.stats().as_array() == stats).all(), (b.stats().as_dict(), stats)
    assert stats[1] > n
    b.close()


@pytest.mark.gpu
@offsets
@pools
def test_offsets_policy_moves(pb, orc, off, nT):
    """pom_batch_policy_moves (its draws come from the RNG of global env off + e) + pom_batch_step with auto-reset"""
    n, ticks, seed, mask = 3000, 60, 76, 0b0111
    b = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=40)
    T, _ = b.templates()
    S, _ = b.download()
    dev = b.alloc(4 * n)
    for t in range(ticks):
        b.generate_moves(dev, seed, t, 6)
        b.policy_moves(dev, seed, t, mask)
        b.step(dev, AR | COUNT)
    A = orc.simple_agents(n)
    status, stats = _oracle_policy_rollout(orc, S, T, A, off, ticks, seed, 6, 40, mask)
    G, gst = b.download()
    _same(orc, G, gst, S, status, "policy")
    assert (b.stats().as_array() == stats).all(), (b.stats().as_dict(), stats)
    assert b.policy_download().tobytes() == A.tobytes()
    b.free(dev)
    b.close()


@pytest.mark.gpu
@offsets
@pools
def test_offsets_tick_wrap(pb, orc, off, nT):
    """a rollout from tick0 = 2^32 - 50 over 100 ticks in two launches (the second starts at tick 0) equals
    generate_moves + step tick by tick and the replay at ticks (tick0 + k) mod 2^32"""
    n, ticks, seed, tick0 = 3000, 100, 77, 2 ** 32 - 50
    a = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=60)
    c = pb.Batch(n, env_offset=off, n_templates=nT, max_ticks=60)
    T, _ = a.templates()
    S, _ = a.download()
    a.rollout(50, seed, tick0, 0)
    a.rollout(50, seed, (tick0 + 50) & U32, 0)
    dev = c.alloc(4 * n)
    for k in range(ticks):
        c.generate_moves(dev, seed, (tick0 + k) & U32, 6)
        c.step(dev, AR | COUNT)
    status, stats = replay(orc, S, T, off, ticks, seed, 6, 60, tick0=tick0)
    for h, what in ((a, "rollout"), (c, "per tick")):
        G, gst = h.download()
        _same(orc, G, gst, S, status, what)
        assert (h.stats().as_array() == stats).all(), (what, h.stats().as_dict(), stats)
    c.free(dev)
    a.close()
    c.close()


# ----------------------------------------------------------------------------------------------------------- D: list


class _ListBuffers:
    """device buffers of pom_batch_step_compact: joint actions, done bits, the finished-env list with GUARD sentinel
    entries behind its end, and its count in device memory or in mapped host memory"""
    GUARD = 64

    def __init__(self, pb, b, cap, mapped_count=False):
        self.pb, self.b, self.n, self.cap = pb, b, b.n, cap
        self.words = (self.n + 31) // 32
        self.joint = b.alloc(2 * self.n)
        self.bits = b.alloc(4 * self.words)
        self.lst = b.alloc(4 * (cap + self.GUARD))
        self.lst_st = b.alloc(cap + self.GUARD)
        self.owner = None
        if mapped_count:
            self.count_host, self.owner = pb.pinned_array((1,), np.uint32)
            self.count = C.c_void_p(self.count_host.ctypes.data)
        else:
            self.count = b.alloc(4)

    def tick(self, joint, capacity, flags=0):
        pb = self.pb
        _to_dev(pb, self.joint, np.ascontiguousarray(joint, np.uint16))
        _to_dev(pb, self.lst, np.full(self.cap + self.GUARD, 0xDEADBEEF, np.uint32))
        _to_dev(pb, self.lst_st, np.full(self.cap + self.GUARD, 0xAB, np.uint8))
        _to_dev(pb, self.bits, np.full(self.words, 0x5A5A5A5A, np.uint32))
        if self.owner is not None:
            self.count_host[0] = 0xFFFFFFFF
        else:
            _to_dev(pb, self.count, np.full(1, 0xFFFFFFFF, np.uint32))
        assert capacity <= self.cap
        io = pb.StepCompactIO(self.joint, self.bits, self.lst, self.lst_st, self.count, capacity, None, 0, 4)
        self.b.step_compact_io(io, flags)
        self.b.sync()
        self.capacity = capacity

    def check(self, ended, status):
        """the list is a permutation of the ended envs (clipped to the capacity: distinct ended envs), each entry with its
        status byte, the count exact, the done bits complete with the tail word's spare bits zero, the guards untouched"""
        pb = self.pb
        count = int(self.count_host[0]) if self.owner is not None else int(_from_dev(pb, np.zeros(1, np.uint32), self.count)[0])
        lst = _from_dev(pb, np.zeros(self.cap + self.GUARD, np.uint32), self.lst)
        lst_st = _from_dev(pb, np.zeros(self.cap + self.GUARD, np.uint8), self.lst_st)
        bits = _from_dev(pb, np.zeros(self.words, np.uint32), self.bits)
        idx = np.nonzero(ended)[0]
        assert count == min(idx.size, self.capacity), (count, idx.size, self.capacity)
        got = lst[:count].astype(np.int64)
        if count == idx.size:
            assert (np.sort(got) == idx).all(), "the list is not a permutation of the ended envs"
        else:
            assert np.unique(got).size == count and ended[np.minimum(got, self.n - 1)].all() and (got < self.n).all()
        assert (lst_st[:count] == status[got]).all()
        assert (lst[count:] == 0xDEADBEEF).all() and (lst_st[count:] == 0xAB).all(), "written past the list's end"
        want = np.zeros(self.words * 32, bool)
        want[:self.n] = ended
        want_words = np.packbits(want, bitorder="little").view("<u4")
        assert (bits == want_words).all(), "done bits, word %d" % np.nonzero(bits != want_words)[0][0]

    def free(self):
        for p in (self.joint, self.bits, self.lst, self.lst_st):
            self.b.free(p)
        if self.owner is not None:
            self.pb.pinned_free(self.owner)
        else:
            self.b.free(self.count)


def _ending_mask(case, n, grid, rng):
    """which envs end in the tick: env e lives in CTA (e // 32) % grid when the walk is forward"""
    cta = (np.arange(n) // 32) % grid
    m = np.zeros(n, bool)
    if case == "all":
        m[:] = True
    elif case == "none":
        pass
    elif case.startswith("cta0-"):
        m[rng.choice(np.nonzero(cta == 0)[0], int(case[5:]), replace=False)] = True
    elif case.startswith("every-"):
        for c in range(grid):
            m[rng.choice(np.nonzero(cta == c)[0], int(case[6:]), replace=False)] = True
    else:                                                           # random, about 480 per CTA on average
        m = rng.random(n) < 480 / 1024
        per = np.bincount(cta[m], minlength=grid)
        assert per.min() < 480 < per.max(), (per.min(), per.max())
    return m


class _ListRig:
    """a handle made with POM_STEP_PINGPONG=0 (forward walk, so the CTA of every slice is known) of SMs x 1024 + 13 envs
    (32 slices per CTA and a ragged tail) and a twin stepped with pom_batch_step_host: fresh templates, with the envs
    that are to end in the next tick uploaded at timeStep 65535"""

    def __init__(self, pb, monkeypatch):
        self.grid = _sm_count()
        self.n = n = self.grid * 1024 + 13
        monkeypatch.setenv("POM_STEP_PINGPONG", "0")
        self.a = pb.Batch(n, n_templates=16, empty=True)
        monkeypatch.delenv("POM_STEP_PINGPONG")
        self.c = pb.Batch(n, n_templates=16, empty=True)
        T, _ = self.a.templates()
        self.S0 = np.ascontiguousarray(T[np.arange(n) % 16])

    def arm(self, ends):
        S = self.S0.copy()
        S["timeStep"][ends] = CEIL
        self.a.upload(S)
        self.c.upload(S)

    def twin(self):
        want = np.zeros(self.n, np.uint8)
        self.c.step_host(np.zeros((self.n, 4), np.uint8), want, 0)
        return want

    def close(self):
        self.a.close()
        self.c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["all", "cta0-480", "cta0-481", "every-480", "every-481", "random"])
def test_finished_list_at_the_cta_capacity(pb, monkeypatch, case):
    """the finished-env list when a CTA's shared list of 480 entries fills exactly and overflows into the global list"""
    R = _ListRig(pb, monkeypatch)
    ends = _ending_mask(case, R.n, R.grid, np.random.default_rng(78))
    R.arm(ends)
    L = _ListBuffers(pb, R.a, R.n)
    L.tick(np.zeros(R.n, np.uint16), R.n)
    want = R.twin()
    assert (((want & ENDED) != 0) == ends).all()
    L.check(ends, want)
    L.free()
    R.close()


@pytest.mark.gpu
@pytest.mark.parametrize("capacity", [1000, 0])
def test_finished_list_clipped_to_capacity(pb, monkeypatch, capacity):
    """a capacity smaller than the buffer: the count is clipped, every entry is a distinct ended env with its status,
    nothing is written past the capacity"""
    R = _ListRig(pb, monkeypatch)
    ends = _ending_mask("every-481", R.n, R.grid, np.random.default_rng(79))
    R.arm(ends)
    L = _ListBuffers(pb, R.a, R.n)
    L.tick(np.zeros(R.n, np.uint16), capacity)
    L.check(ends, R.twin())
    L.free()
    R.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mapped_count", [False, True], ids=["device-count", "mapped-count"])
def test_finished_list_counter_reset(pb, monkeypatch, mapped_count):
    """the counter behind the list starts from zero in every launch: a clipped tick, an overflowing tick, a tick that
    ends nothing and a full-list tick each report exactly their own list"""
    R = _ListRig(pb, monkeypatch)
    rng = np.random.default_rng(80)
    L = _ListBuffers(pb, R.a, R.n, mapped_count)
    for case, capacity in (("every-481", 1000), ("every-481", R.n), ("none", R.n), ("all", R.n)):
        ends = _ending_mask(case, R.n, R.grid, rng)
        R.arm(ends)
        L.tick(np.zeros(R.n, np.uint16), capacity)
        L.check(ends, R.twin())
    L.free()
    R.close()
