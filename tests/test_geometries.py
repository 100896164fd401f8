"""The step path outside the batch sizes and the kernel geometry the rest of the suite runs, against the oracle:
  A  batches of 4 Mi + 1500 envs on the default geometry: every CTA of k_step_ws takes more than 3 x 256 slices, so the
     256-entry mail ring that hands slices from the producer warp to the compute warps wraps several times, and the
     observation slabs of four agents pass 4 GiB of byte offsets;
  B  every kernel image and host path that a tuning switch selects (POM_TPB, POM_WS_NW, POM_WS_NOSPEC, POM_STEP_PARTS,
     POM_CHUNKS, POM_ZEROCOPY; INTEGRATION section 6);
  C  proof that each configuration ran the code it names: launches per call for the host-side switches (each switch set
     after another handle has already stepped in the same process: the switches are read per handle), and the template
     arguments of the kernels that a torch.profiler trace lists for the kernel images.
Every comparison is field by field (orc.diff_batch) plus the status bytes, and all ten counters where the whole batch is
replayed.  The big batches are replayed in windows of at most 128 Ki envs on a thread pool (replay_windows): envs are
independent, and no whole-batch array of states is ever held on the host (one would take 4.2 GB).  The CPU test checks
the windowed replay against test_gpu_parity._oracle_rollout."""
import ctypes as C
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from test_gpu_parity import _oracle_rollout
from test_gpu_policy import _oracle_policy_rollout
from test_limits import (AR, COUNT, DONE, ENDED, INVALID, Replay, _ListBuffers, _ListRig, _ending_mask, _from_dev,
                         _oracle_templates, _sm_count, ceiling_step, raw_step, replay)
from test_rewards import reward_definition
from test_teams import team_orc  # noqa: F401  (fixture: the team game on the restatement)

RAW, OVERLAP = 0x1, 0x8
MAIL = 256                       # RingScratch::MAIL: the mail ring of k_step_ws
WINDOW = 1 << 17
NT = 64                          # templates of every handle here
MT = 42                          # max_ticks of the stepped handles: reached inside a few ticks from the mid-game states
PREROLL = 40                     # ticks of the fused rollout that makes the mid-game states


# ----------------------------------------------------------------------------------------------------------- windows


def windows(n, size=WINDOW):
    """[(first, count)] covering envs 0..n-1"""
    return [(f, min(size, n - f)) for f in range(0, n, size)]


def replay_windows(job, wins):
    """job(first, count) for every window on a thread pool (the oracle's ctypes calls release the GIL); results in
    window order"""
    with ThreadPoolExecutor(max(1, min(8, os.cpu_count() or 1))) as ex:
        return list(ex.map(lambda w: job(*w), wins))


def ring_windows(n, grid):
    """the env windows whose slices are tickets 255..257 of every CTA of a whole-batch k_step_ws launch (ticket t of CTA
    c is slice c + t * grid, mirrored on the ticks that walk the batch backwards), and the first and last slices"""
    ns = (n + 31) // 32
    out = [(0, 32), ((ns - 1) * 32, n - (ns - 1) * 32)]
    lo, hi = (MAIL - 1) * grid, (MAIL + 2) * grid                       # slices [lo, hi) forward
    for a, b in ((lo, hi), (ns - hi, ns - lo)):                         # and mirrored
        out.append((a * 32, min(b * 32, n) - a * 32))
    return sorted(out)


# ----------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("no_reset", [False, True], ids=["reset", "no-reset"])
def test_windowed_replay_matches_oracle_rollout(orc, no_reset):
    """Replay run window by window on the thread pool == _oracle_rollout on the whole batch: every field, the status
    bytes and the summed counters; ragged windows, resets from the pool by global env index, truncation"""
    n, ticks, seed, nT, mt = 1003, 90, 17, 24, 40
    T = _oracle_templates(orc, nT)
    S0 = T[np.arange(n) % nT].copy()
    A = S0.copy()
    st_a, stats_a = _oracle_rollout(orc, A, T, 0, ticks, seed, 6, mt, no_reset=no_reset)

    def job(f, c):
        R = Replay(orc, S0[f:f + c].copy(), T, f, mt, no_reset)
        for t in range(ticks):
            R.tick(orc.rng_moves(seed, f, c, t, 6))
        return R

    rs = replay_windows(job, windows(n, 96))
    B = np.concatenate([r.S for r in rs])
    assert orc.diff_batch(A, B)[0] == -1
    assert (np.concatenate([r.status for r in rs]) == st_a).all()
    assert (sum(r.stats for r in rs) == stats_a).all()
    assert stats_a[7] > 0 and stats_a[1] > stats_a[7]


def test_ring_windows_cover_the_wrapping_tickets():
    """ring_windows holds, for every CTA and both walk directions, the slices of tickets 255..257"""
    grid, n = 148, (4 << 20) + 1500
    ns = (n + 31) // 32
    W = ring_windows(n, grid)
    covered = np.zeros(ns, bool)
    for f, c in W:
        assert f % 32 == 0 and c > 0 and f + c <= n
        covered[f // 32:(f + c + 31) // 32] = True
    for t in (255, 256, 257):
        s = np.arange(grid) + t * grid
        assert covered[s].all() and covered[ns - 1 - s].all()
    assert covered[0] and covered[-1]


# ----------------------------------------------------------------------------------------------------------- GPU helpers


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


def _mid_game(pb, n, seed=5151):
    """n running mid-game states: fresh templates rolled PREROLL ticks forward by the fused rollout (pinned to the oracle
    elsewhere) on the default geometry; returned as the source handle, which keeps them"""
    src = pb.Batch(n, n_templates=NT)
    src.rollout(PREROLL, seed, 0, 0)
    return src


def _fresh(pb, src, n, env0=0, teams=False, max_ticks=MT):
    """a fresh handle (episode numbers zero, as Replay assumes) with the same template pool, holding src's states"""
    b = pb.Batch(n, env_offset=env0, n_templates=NT, max_ticks=max_ticks, empty=True, teams=teams)
    for f, c in windows(n, 1 << 20):
        b.upload(src.download(f, c)[0], first=f)
    return b


def _same(orc, G, gst, S, st, what):
    e, why = orc.diff_batch(G, S)
    assert e == -1, "%s: env %d field group %d" % (what, e, why)
    bad = np.nonzero(gst != st)[0]
    assert bad.size == 0, "%s: status of env %d: %#x != %#x" % (what, bad[0], gst[bad[0]], st[bad[0]])


def _stats_ok(got, want):
    """all ten counters equal, and the ticks saw game ends and truncations"""
    assert (got == want).all(), (got, want)
    assert want[1] > want[7] > 0 and want[2:7].sum() > 0


class Locked:
    """one handle's transfers from several threads: pom_batch_download stages through per-handle buffers"""

    def __init__(self, b):
        self.b, self.lock = b, threading.Lock()

    def download(self, f, c):
        with self.lock:
            return self.b.download(f, c)


# ----------------------------------------------------------------------------------------------------------- A: big batches


BIG = (4 << 20) + 1500
BIG_PATHS = ["spec", "frozen-misaligned", "raw-misaligned", "overlap", "step_host", "compact", "rewards", "observe",
             "team", "simple"]
FULL = ("spec", "overlap")       # replayed in full: their counters are compared


@pytest.fixture(scope="module")
def big_src(pb):
    src = _mid_game(pb, BIG)
    yield src
    src.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", BIG_PATHS)
def test_big_batch(pb, orc, team_orc, big_src, path):
    """4 Mi + 1500 envs from mid-game states, a few ticks in both walk directions.  spec: the plain loop AUTORESET |
    COUNT (SPEC image); frozen / raw: flags 0 and POM_STEP_RAW with moves 4 bytes off 16-byte alignment (the generic
    image, per-lane move loads); overlap: POM_STEP_OVERLAP (two persistent parts); step_host: pinned buffers (zero-copy
    status bytes); compact: done bits and a finished list of capacity n; rewards: step_rewards; observe: step_observe
    with agent_mask 15 (slabs 2 and 3 start past 4 GiB); team: a team handle's plain loop; simple: a SimpleAgent rollout
    (tick by tick at this size: k_policy_moves and the FREEZE image).  spec and overlap are replayed in full, the others
    on ring_windows."""
    n, seed, ticks = BIG, 88, 4
    grid = _sm_count()
    ns = (n + 31) // 32
    assert ns / grid > 3 * MAIL
    if path == "overlap":
        per = ((n + 1) // 2 + 1023) // 1024 * 1024
        for count in (per, n - per):
            assert (count + 31) // 32 / grid > MAIL
    o = team_orc if path == "team" else orc
    b = _fresh(pb, big_src, n, teams=path == "team")
    T, _ = b.templates()
    flags = {"frozen-misaligned": 0, "raw-misaligned": RAW, "compact": 0, "observe": 0}.get(path, AR | COUNT)
    wins = windows(n) if path in FULL else ring_windows(n, grid)
    outs = {w: [] for w in wins}                                    # per-tick outputs of the windows
    dev = b.alloc(4 * n + 16)
    mv_ptr = dev.value + (4 if path.endswith("misaligned") else 0)
    owners, obs = [], None
    if path == "step_host":
        mvp, o1 = pb.pinned_array((n, 4), np.uint8)
        out, o2 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2]
    elif path == "rewards":
        rw, o1 = pb.pinned_array((n, 4), np.int8)
        out, o2 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2]
    elif path == "compact":
        L = _ListBuffers(pb, b, n)
    elif path == "observe":
        stride = int(pb.lib().pom_batch_obs_stride(b.h))
        assert 2 * stride * pb.OBS_BYTES > 1 << 32
        obs = b.alloc(4 * stride * pb.OBS_BYTES)
    if path == "simple":
        l0 = b.launch_count()
        b.rollout(ticks, seed, 0, pb.ROLL_SIMPLE(15))
        assert b.launch_count() - l0 == 2 * ticks
    for t in range(ticks):
        if path == "step_host":
            mvp[:] = orc.rng_moves(seed, 0, n, t, 6)
            b.step_host(mvp, out, flags)
        elif path == "compact":
            before = b.status()
            L.tick(pb.joint_of_moves(orc.rng_moves(seed, 0, n, t, 6)), n, flags)
            after = b.status()
            L.check(((before & (DONE | INVALID)) == 0) & ((after & ENDED) != 0), after)
            out = after
        elif path != "simple":
            b.generate_moves(mv_ptr, seed, t, 6)
            if path == "rewards":
                b.step_rewards(mv_ptr, rw, out, flags)
                b.sync()
            elif path == "observe":
                b.step_observe(mv_ptr, obs, 15, 4, flags)
            else:
                b.step(mv_ptr, flags | (OVERLAP if path == "overlap" else 0))
        for f, c in wins:
            if path in ("step_host", "compact"):
                outs[(f, c)].append(out[f:f + c].copy())
            elif path == "rewards":
                outs[(f, c)].append((out[f:f + c].copy(), rw[f:f + c].copy()))
    B = Locked(b)
    S0 = Locked(big_src)
    planes = {}
    if path == "observe":
        b.sync()
        for k in range(4):
            for f, c in wins:
                planes[(k, f)] = _from_dev(pb, np.zeros((c, pb.OBS_BYTES), np.uint8),
                                           C.c_void_p(obs.value + (k * stride + f) * pb.OBS_BYTES))

    def job(f, c):
        S, _ = S0.download(f, c)
        if path == "simple":
            A = orc.simple_agents(c)
            status, stats = _oracle_policy_rollout(orc, S, T, A, f, ticks, seed, 6, MT, 15)
            G, gst = B.download(f, c)
            _same(orc, G, gst, S, status, "simple [%d, %d)" % (f, f + c))
            with B.lock:
                assert b.policy_download(f, c).tobytes() == A.tobytes(), "agent memories [%d, %d)" % (f, f + c)
            return stats
        R = Replay(o, S, T, f, MT)
        for t in range(ticks):
            mv = orc.rng_moves(seed, f, c, t, 6)
            stepped = (R.status & (DONE | INVALID)) == 0
            if path == "raw-misaligned":
                raw_step(orc, R.S, R.status, mv)
                end = R.status.copy()
            else:
                end = R.tick(mv, autoreset=bool(flags & AR))
            if path in ("step_host", "compact"):
                got = outs[(f, c)][t]
                assert (got == end).all(), "tick %d: status of env %d" % (t, f + np.nonzero(got != end)[0][0])
            elif path == "rewards":
                gst, grw = outs[(f, c)][t]
                assert (gst == end).all(), "tick %d: status of env %d" % (t, f + np.nonzero(gst != end)[0][0])
                want = reward_definition(stepped, end, R.S["agents"]["dead"] != 0, False)
                assert (grw == want).all(), "tick %d: rewards of env %d" % (t, f + np.nonzero((grw != want).any(1))[0][0])
        G, gst = B.download(f, c)
        _same(orc, G, gst, R.S, R.status, "%s [%d, %d)" % (path, f, f + c))
        for k in range(4 if path == "observe" else 0):
            want = orc.observe_planes_batch(R.S, k, 4)
            got = planes[(k, f)]
            assert (got == want).all(), "agent %d planes of env %d" % (k, f + np.nonzero((got != want).any(1))[0][0])
        return R.stats

    stats = sum(replay_windows(job, wins))
    if path in FULL:
        _stats_ok(b.stats().as_array(), stats)
    elif not flags & AR and path != "simple":
        assert not b.stats().as_array().any()
    assert stats[1] > 0 or not flags & AR
    b.free(dev)
    if obs is not None:
        b.free(obs)
    if path == "compact":
        L.free()
    for x in owners:
        pb.pinned_free(x)
    b.close()


# ----------------------------------------------------------------------------------------------------------- B: switches


def _switched(pb, monkeypatch, env, n, src=None, env0=0, teams=False):
    """a handle made with the switches `env` set, holding mid-game states (made on the default geometry before the
    switches are set); returns (handle, states, templates)"""
    own = src is None
    src = _mid_game(pb, n) if own else src
    S, _ = src.download()
    if own:
        src.close()
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    b = pb.Batch(n, env_offset=env0, n_templates=NT, max_ticks=MT, empty=True, teams=teams)
    for k in env:
        monkeypatch.delenv(k)
    b.upload(S)
    return b, S, b.templates()[0]


def _stats_check(b, R, flags):
    got = b.stats().as_array()
    if flags & AR:
        want = R.stats.copy()
        if not flags & COUNT:
            want[0] = 0
        _stats_ok(got, want)
    else:
        assert not got.any()


def _per_tick_check(pb, orc, b, S, T, env0, flags, ticks, seed, how="step"):
    n = b.n
    R = Replay(orc, S, T, env0, MT)
    dev = b.alloc(4 * n)
    owners = []
    if how == "pinned":
        mv, o1 = pb.pinned_array((n, 4), np.uint8)
        out, o2 = pb.pinned_array((n,), np.uint8)
        owners = [o1, o2]
    else:
        mv, out = None, np.zeros(n, np.uint8)
    launches = []
    for t in range(ticks):
        m = orc.rng_moves(seed, env0, n, t, 6)
        if how == "step":
            b.generate_moves(dev, seed, t, 6)
            l0 = b.launch_count()
            b.step(dev, flags)
        else:
            l0 = b.launch_count()
            if mv is not None:
                mv[:] = m
            b.step_host(m if mv is None else mv, out, flags)
        b.sync()
        launches.append(b.launch_count() - l0)
        if flags & RAW:
            raw_step(orc, R.S, R.status, m)
            end = R.status
        else:
            end = R.tick(m, autoreset=bool(flags & AR))
        if how != "step":
            assert (out == end).all(), "tick %d: status of env %d" % (t, np.nonzero(out != end)[0][0])
    G, gst = b.download()
    _same(orc, G, gst, R.S, R.status, "after %d ticks" % ticks)
    _stats_check(b, R, flags)
    b.free(dev)
    for o in owners:
        pb.pinned_free(o)
    return launches


TPB_PATHS = ["tile-0", "tile-autoreset", "tile-raw", "overlap", "rollout", "harmless", "no_reset", "step_seq",
             "simple", "policy_moves", "planes", "cropped", "expand"]


@pytest.mark.gpu
@pytest.mark.parametrize("path", TPB_PATHS)
@pytest.mark.parametrize("tpb", [32, 64, 256])
def test_tpb_images(pb, orc, monkeypatch, tpb, path):
    """POM_TPB: the free-for-all k_step<TPB> (POM_STEP_KERNEL=tile with flags 0 / AUTORESET | COUNT / RAW; the two
    overlap parts at 2^18 + 1500 envs), k_rollout<TPB> (SPEC, HARMLESS, NO_RESET, step_seq, SimpleAgents),
    k_policy_moves<TPB>, k_observe_planes<TPB> (full at views 0, 4, 10; cropped at 0, 4, 5) and k_expand_step<TPB>
    (fanouts 1, 7, 1296 and the envs behind a partial last slice) against the oracle"""
    n = (1 << 18) + 1500 if path == "overlap" else 3001
    env0, seed = 77, 300 + tpb
    env = {"POM_TPB": tpb}
    if path.startswith("tile"):
        env["POM_STEP_KERNEL"] = "tile"
    b, S, T = _switched(pb, monkeypatch, env, n, env0=env0)
    if path.startswith("tile"):
        flags = {"tile-0": 0, "tile-autoreset": AR | COUNT, "tile-raw": RAW}[path]
        assert _per_tick_check(pb, orc, b, S, T, env0, flags, 24, seed) == [1] * 24
    elif path == "overlap":
        dev = b.alloc(4 * n)
        R = Replay(orc, S, T, env0, MT)
        for t in range(8):
            b.generate_moves(dev, seed, t, 6)
            l0 = b.launch_count()
            b.step(dev, AR | COUNT | OVERLAP)
            assert b.launch_count() - l0 == 2
            R.tick(orc.rng_moves(seed, env0, n, t, 6))
        G, gst = b.download()
        _same(orc, G, gst, R.S, R.status, "overlap")
        _stats_ok(b.stats().as_array(), R.stats)
        b.free(dev)
    elif path in ("rollout", "harmless", "no_reset", "step_seq"):
        ticks = 60
        if path == "step_seq":
            seq = b.alloc(4 * n * ticks)
            for t in range(ticks):
                b.generate_moves(seq.value + 4 * n * t, seed, t, 6)
            b.step_seq(seq, ticks, 0)
            b.free(seq)
        else:
            b.rollout(ticks, seed, 0, {"rollout": 0, "harmless": pb.ROLL_HARMLESS, "no_reset": pb.ROLL_NO_RESET}[path])
        status, stats = replay(orc, S, T, env0, ticks, seed, 5 if path == "harmless" else 6, MT,
                               no_reset=path == "no_reset")
        G, gst = b.download()
        _same(orc, G, gst, S, status, path)
        _stats_ok(b.stats().as_array(), stats)
    elif path == "simple":
        A = orc.simple_agents(n)
        b.rollout(50, seed, 0, pb.ROLL_SIMPLE(15))
        status, stats = _oracle_policy_rollout(orc, S, T, A, env0, 50, seed, 6, MT, 15)
        G, gst = b.download()
        _same(orc, G, gst, S, status, path)
        assert (b.stats().as_array() == stats).all() and stats[1] > 0
        assert b.policy_download().tobytes() == A.tobytes()
    elif path == "policy_moves":
        A = orc.simple_agents(n)
        status = np.zeros(n, np.uint8)
        for t in range(30):
            mv = orc.rng_moves(seed, env0, n, t, 6)
            gm = mv.copy()
            b.policy_moves_host(gm, seed, t, 0b1011)
            orc.simple_moves_batch(S, status, A, seed, env0, t, 0b1011, mv)
            live = (status & (DONE | INVALID)) == 0
            assert (gm[live] == mv[live]).all(), "tick %d: moves of env %d" % (t, np.nonzero((gm != mv).any(1) & live)[0][0])
            b.step_host(gm, None, 0)
            fl = np.zeros(n, np.uint8)
            orc.env_step_batch(S, status, mv, fl)
            status[(fl & 0x3E) != 0] |= INVALID
        G, gst = b.download()
        _same(orc, G, gst, S, status, path)
        assert b.policy_download().tobytes() == A.tobytes()
    elif path in ("planes", "cropped"):
        for view in ((0, 4, 10) if path == "planes" else (0, 4, 5)):
            got = b.observe_planes(0b1101, view) if path == "planes" else b.observe_planes_cropped(0b1101, view)
            for k, agent in enumerate((0, 2, 3)):
                want = (orc.observe_planes_batch(S, agent, view) if path == "planes" else
                        orc.observe_cropped_batch(S, agent, view))
                bad = np.nonzero((got[k] != want).any(1))[0]
                assert bad.size == 0, "view %d agent %d env %d" % (view, agent, bad[:1])
    else:
        _expand_check(pb, orc, b, S, monkeypatch, env)
    b.close()


def _expand_check(pb, orc, src, S, monkeypatch, env):
    """k_expand_step of the destination handle's geometry (made with the switches `env`): every child of roots at
    fanouts 1, 7 and 1296, and a partial last slice that must leave the destination's envs behind it alone"""
    st0 = src.status()
    for fanout, roots in ((1, np.arange(0, 3001, 37)), (7, np.arange(5, 3001, 211)), (1296, np.array([3, 2999]))):
        roots = roots.astype(np.uint32)
        m = roots.size * fanout + 45                                # envs behind the children
        for k, v in env.items():
            monkeypatch.setenv(k, str(v))
        dst = pb.Batch(m, n_templates=NT)
        for k in env:
            monkeypatch.delenv(k)
        before, sb = dst.download()
        dst.expand_step_from(src, roots, fanout, 0)
        G, gst = dst.download()
        k = roots.size * fanout
        assert G[k:].tobytes() == before[k:].tobytes() and (gst[k:] == sb[k:]).all(), "fanout %d: envs behind" % fanout
        j = np.tile(np.arange(fanout), roots.size)
        mv = np.ascontiguousarray(np.stack([j % 6, (j // 6) % 6, (j // 36) % 6, (j // 216) % 6], axis=1).astype(np.uint8))
        E = np.repeat(S[roots], fanout)
        est = np.repeat(st0[roots], fanout)
        orc.env_step_batch(E, est, mv)
        _same(orc, G[:k], gst[:k], E, est, "fanout %d" % fanout)
        dst.close()


NW_PATHS = ["step-0", "step-autoreset", "step_host", "compact"]


@pytest.mark.gpu
@pytest.mark.parametrize("path", NW_PATHS)
@pytest.mark.parametrize("nw", [12, 14, 16, 18, 22])
def test_ws_nw_images(pb, orc, monkeypatch, nw, path):
    """POM_WS_NW: k_step_ws<NW> (the generic image, no observations) on SMs x 40 slices + 1500 envs (every one of the
    24 slice buffers of a CTA reused): flags 0 / AUTORESET | COUNT, step_host with pinned buffers, and step_compact with
    a finished list that overflows the 480 entries a CTA keeps in shared memory"""
    grid = _sm_count()
    seed, env0 = 400 + nw, 31
    if path == "compact":
        monkeypatch.setenv("POM_WS_NW", str(nw))
        R = _ListRig(pb, monkeypatch)
        monkeypatch.delenv("POM_WS_NW")
        ends = _ending_mask("every-481", R.n, R.grid, np.random.default_rng(nw))
        R.arm(ends)
        S = R.S0.copy()
        S["timeStep"][ends] = 65535
        L = _ListBuffers(pb, R.a, R.n)
        mv = orc.rng_moves(seed, 0, R.n, 0, 6)
        L.tick(pb.joint_of_moves(mv), R.n)
        st = np.zeros(R.n, np.uint8)
        ceiling_step(orc, S, st, mv)
        L.check((st & ENDED) != 0, st)
        G, gst = R.a.download()
        _same(orc, G, gst, S, st, "compact")
        assert ((st & ENDED) != 0).sum() >= 481 * grid
        L.free()
        R.close()
        return
    n = grid * 32 * 40 + 1500
    b, S, T = _switched(pb, monkeypatch, {"POM_WS_NW": nw}, n, env0=env0)
    if path == "step_host":
        _per_tick_check(pb, orc, b, S, T, env0, AR | COUNT, 6, seed, "pinned")
    else:
        _per_tick_check(pb, orc, b, S, T, env0, 0 if path == "step-0" else AR | COUNT, 6, seed)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["plain", "rollout", "overlap"])
def test_ws_nospec(pb, orc, monkeypatch, path):
    """POM_WS_NOSPEC=1: the generic images in the plain loop and the headline rollout, and POM_STEP_OVERLAP at
    2^18 + 1500 envs on the persistent kernel instead of the tile kernel"""
    n = (1 << 18) + 1500 if path == "overlap" else 5003
    seed, env0 = 500, 9
    b, S, T = _switched(pb, monkeypatch, {"POM_WS_NOSPEC": 1}, n, env0=env0)
    if path == "rollout":
        b.rollout(60, seed, 0, 0)
        status, stats = replay(orc, S, T, env0, 60, seed, 6, MT)
        G, gst = b.download()
        _same(orc, G, gst, S, status, path)
        _stats_ok(b.stats().as_array(), stats)
    else:
        dev = b.alloc(4 * n)
        R = Replay(orc, S, T, env0, MT)
        for t in range(30 if path == "plain" else 8):
            b.generate_moves(dev, seed, t, 6)
            b.step(dev, AR | COUNT | (OVERLAP if path == "overlap" else 0))
            R.tick(orc.rng_moves(seed, env0, n, t, 6))
        G, gst = b.download()
        _same(orc, G, gst, R.S, R.status, path)
        _stats_ok(b.stats().as_array(), R.stats)
        b.free(dev)
    b.close()


def _warm(pb, n, how):
    """a handle of the default configuration that has already stepped (overlap, step_host pageable or pinned): a switch
    set after this must still be read by the next handle"""
    w = pb.Batch(n, n_templates=8)
    if how == "overlap":
        dev = w.alloc(4 * n)
        w.generate_moves(dev, 1, 0, 6)
        w.step(dev, OVERLAP)
        w.sync()
        w.free(dev)
    elif how == "pinned":
        mv, o1 = pb.pinned_array((n, 4), np.uint8)
        w.step_host(mv, None, 0)
        pb.pinned_free(o1)
    else:
        w.step_host(np.zeros((n, 4), np.uint8), None, 0)
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [(1 << 18) + 1500, (1 << 19) + 1500], ids=["tile-parts", "persistent-parts"])
@pytest.mark.parametrize("parts", [3, 16])
def test_step_parts(pb, orc, monkeypatch, parts, n):
    """POM_STEP_PARTS: overlap with more than two parts, on both sides of 0.5 Mi envs; `parts` launches per step, with
    the switch set after another handle has already stepped with POM_STEP_OVERLAP"""
    _warm(pb, 1 << 18, "overlap")
    seed, env0 = 600 + parts, 0
    b, S, T = _switched(pb, monkeypatch, {"POM_STEP_PARTS": parts}, n, env0=env0)
    per = ((n + parts - 1) // parts + 1023) // 1024 * 1024
    want = -(-n // per)
    assert want > 2
    dev = b.alloc(4 * n)
    R = Replay(orc, S, T, env0, MT)
    for t in range(8):
        b.generate_moves(dev, seed, t, 6)
        l0 = b.launch_count()
        b.step(dev, AR | COUNT | OVERLAP)
        assert b.launch_count() - l0 == want
        R.tick(orc.rng_moves(seed, env0, n, t, 6))
    G, gst = b.download()
    _same(orc, G, gst, R.S, R.status, "parts")
    _stats_ok(b.stats().as_array(), R.stats)
    b.free(dev)
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunks,zerocopy", [(1, 1), (5, 1), (16, 1), (6, 0)], ids=["chunks-1", "chunks-5", "chunks-16",
                                                                                 "zerocopy-0"])
def test_step_host_pipeline_switches(pb, orc, monkeypatch, chunks, zerocopy):
    """POM_CHUNKS with pageable buffers at 300,000 envs, and POM_ZEROCOPY=0 with pinned buffers (the copy pipeline instead
    of the kernel reading host memory); the chunks per step_host, with the switch set after another handle has already
    taken the same path"""
    n, seed, env0 = 300_000, 700 + chunks, 3
    how = "pageable" if zerocopy else "pinned"
    _warm(pb, 1 << 18, how)
    env = {"POM_CHUNKS": chunks} if zerocopy else {"POM_ZEROCOPY": 0}
    b, S, T = _switched(pb, monkeypatch, env, n, env0=env0)
    per = ((n + chunks - 1) // chunks + 1023) // 1024 * 1024
    launches = _per_tick_check(pb, orc, b, S, T, env0, AR | COUNT, 8, seed, how)
    assert launches == [-(-n // per)] * 8
    b.close()


# ----------------------------------------------------------------------------------------------------------- C: images


@pytest.mark.gpu
def test_zero_copy_is_one_launch(pb, monkeypatch):
    """step_host with pinned buffers: one launch (the kernel reads the moves and writes the status bytes itself), also
    when an earlier handle of the process was made with POM_ZEROCOPY=0 and stepped"""
    n = 300_000
    monkeypatch.setenv("POM_ZEROCOPY", "0")
    _warm(pb, n, "pinned")
    monkeypatch.delenv("POM_ZEROCOPY")
    b = pb.Batch(n, n_templates=8)
    mv, o1 = pb.pinned_array((n, 4), np.uint8)
    l0 = b.launch_count()
    b.step_host(mv, None, 0)
    assert b.launch_count() - l0 == 1
    pb.pinned_free(o1)
    b.close()


IMAGES = [
    # (switches, call, a substring every run of the call must show among its kernels)
    ({"POM_TPB": 32, "POM_STEP_KERNEL": "tile"}, "step", "k_step<32,"),
    ({"POM_TPB": 64, "POM_STEP_KERNEL": "tile"}, "step", "k_step<64,"),
    ({"POM_TPB": 256, "POM_STEP_KERNEL": "tile"}, "step", "k_step<256,"),
    ({"POM_TPB": 32}, "rollout", "k_rollout<32, false, true"),
    ({"POM_TPB": 64}, "rollout_harmless", "k_rollout<64, false, false"),
    ({"POM_TPB": 256}, "rollout_simple", "k_rollout<256, true,"),
    ({"POM_TPB": 32}, "policy_moves", "k_policy_moves<32,"),
    ({"POM_TPB": 256}, "planes", "k_observe_planes<256, false"),
    ({"POM_TPB": 64}, "cropped", "k_observe_planes<64, true"),
    ({"POM_TPB": 32}, "expand", "k_expand_step<32,"),
    ({"POM_WS_NW": 12}, "step", "k_step_ws<12,"),
    ({"POM_WS_NW": 14}, "step", "k_step_ws<14,"),
    ({"POM_WS_NW": 16}, "step", "k_step_ws<16,"),
    ({"POM_WS_NW": 18}, "step", "k_step_ws<18,"),
    ({"POM_WS_NW": 22}, "step", "k_step_ws<22,"),
    ({"POM_WS_NOSPEC": 1}, "plain", "k_step_ws<20, 24, false, false, false"),
    ({}, "plain", "k_step_ws<20, 24, false, false, true"),
    ({"POM_WS_NOSPEC": 1}, "rollout", "k_rollout<128, false, false"),
    ({}, "rollout", "k_rollout<128, false, true"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("env,call,want", IMAGES, ids=["%s-%s" % ("-".join("%s=%s" % kv for kv in e.items()) or "default", c)
                                                        for e, c, _ in IMAGES])
def test_switch_runs_its_image(pb, monkeypatch, env, call, want):
    """each switch configuration runs the kernel image it names: the template arguments of the kernels that
    torch.profiler lists for one call"""
    torch = pytest.importorskip("torch")
    from torch.profiler import ProfilerActivity, profile
    n = 4096
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    b = pb.Batch(n, n_templates=16)
    dst = pb.Batch(4 * 36, n_templates=1, empty=True) if call == "expand" else None     # its geometry runs the expansion
    for k in env:
        monkeypatch.delenv(k)
    b.rollout(10, 3, 0, pb.ROLL_NO_RESET)
    dev = b.alloc(4 * n)
    b.generate_moves(dev, 1, 0, 6)
    b.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        if call == "step":
            b.step(dev, 0)
        elif call == "plain":
            b.step(dev, AR | COUNT)
        elif call == "rollout":
            b.rollout(4, 3, 0, 0)
        elif call == "rollout_harmless":
            b.rollout(4, 3, 0, pb.ROLL_HARMLESS)
        elif call == "rollout_simple":
            b.rollout(4, 3, 0, pb.ROLL_SIMPLE(15))
        elif call == "policy_moves":
            b.policy_moves(dev, 3, 0, 15)
        elif call == "planes":
            b.observe_planes(1, 4)
        elif call == "cropped":
            b.observe_planes_cropped(1, 4)
        elif call == "expand":
            dst.expand_step_from(b, np.arange(4, dtype=np.uint32), 36, 0)
        b.sync()
        if dst is not None:
            dst.sync()
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events() if "pomk::" in e.name})
    assert names, "the profiler lists none of this library's kernels"
    assert any(want in x for x in names), (want, names)
    b.free(dev)
    if dst is not None:
        dst.close()
    b.close()
