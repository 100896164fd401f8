"""pomcpp_b200 — thin ctypes view of the C ABI in include/pom_batch.h (libpom_b200.so).

The product is the shared library (CUDA kernels + C ABI, pomcpp_b200/csrc) and the C++ host layer
(pomcpp_b200/host).  This module only exists so that tests/, bench.py and __graft_entry__.py can call
the ABI from Python; it adds no logic and has NO fallback: if the library is missing, or no CUDA
device is present, the calls raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POM_B200_LIB") or os.path.join(HERE, "libpom_b200.so")   # POM_B200_LIB: A/B runs of two builds

REC_BYTES = 292
OBS_BYTES = 512
ALGO_BYTES_PER_ENV_STEP = 2 * 289 + 4      # SURVEY §8d: packed PAYLOAD in + out + 4 move bytes (what the roofline credits)
MOVED_BYTES_PER_ENV_STEP = 2 * 292 + 4     # what actually crosses HBM: the record is padded to 292 B

STEP_RAW, STEP_AUTORESET, STEP_COUNT, STEP_OVERLAP, STEP_CONTINUE_UNDEFINED = 1, 2, 4, 8, 16
ROLL_HARMLESS, ROLL_NO_RESET, ROLL_CONTINUE_UNDEFINED = 1, 2, 4


def ROLL_SIMPLE(agent_mask):
    """rollout flag: the agents in agent_mask (bit a) play the reference's SimpleAgent"""
    return (agent_mask & 0xF) << 8


INIT_EMPTY, INIT_TEAMS, INIT_RADIO = 1, 2, 4

STATUS_DONE, STATUS_DRAW, STATUS_INVALID, STATUS_TRUNCATED = 0x01, 0x02, 0x10, 0x20

AGENT_DT = np.dtype([("x", "<i4"), ("y", "<i4"), ("bombCount", "<i4"), ("maxBombCount", "<i4"),
                     ("bombStrength", "<i4"), ("canKick", "u1"), ("dead", "u1"), ("_pad", "u1", (2,))])
FLAME_DT = np.dtype([("x", "<i4"), ("y", "<i4"), ("timeLeft", "<i4"), ("strength", "<i4")])
STATE_DT = np.dtype([("board", "<i4", (11, 11)), ("timeStep", "<i4"), ("aliveAgents", "<i4"),
                     ("agents", AGENT_DT, (4,)), ("bombs", "<i4", (20,)), ("bombs_index", "<i4"),
                     ("bombs_count", "<i4"), ("flames", FLAME_DT, (20,)), ("flames_index", "<i4"),
                     ("flames_count", "<i4")])
assert STATE_DT.itemsize == 1004
# include/pom_state.h pom_simple_agent
SIMPLE_DT = np.dtype([("recent", "u1", (4,)), ("rp_index", "u1"), ("rp_count", "u1"), ("move_queue", "<u2")])
assert SIMPLE_DT.itemsize == 8


class InitDesc(C.Structure):
    _fields_ = [("env_offset", C.c_uint64), ("n_templates", C.c_uint32), ("first_seed", C.c_int32),
                ("host_templates", C.c_void_p), ("max_ticks", C.c_uint32), ("flags", C.c_uint32)]


class StepCompactIO(C.Structure):
    _fields_ = [("joint", C.c_void_p), ("done_bits", C.c_void_p), ("fin_env", C.c_void_p), ("fin_status", C.c_void_p),
                ("fin_count", C.c_void_p), ("fin_capacity", C.c_uint32), ("obs_dev", C.c_void_p),
                ("obs_agent_mask", C.c_uint32), ("obs_view", C.c_int32)]


def pack_messages(words):
    """[n, 4, 2] radio words (w0, w1 of agent a, each 0..7) -> [n, 4] uint8 in the encoding of pom_batch_step_radio:
    byte a = w0 | w1 << 3"""
    w = np.asarray(words, np.uint8).reshape(-1, 4, 2)
    return ((w[:, :, 0] & 7) | ((w[:, :, 1] & 7) << 3)).astype(np.uint8)


def unpack_messages(msgs):
    """[n, 4] message bytes -> [n, 4, 2] words (w0, w1); bits 6..7 are ignored, as the device ignores them"""
    m = np.asarray(msgs, np.uint8).reshape(-1, 4)
    return np.stack([m & 7, (m >> 3) & 7], axis=-1).astype(np.uint8)


def joint_of_moves(moves):
    """[n, 4] moves (0..5) -> uint16 joint actions j = a0 + 6 a1 + 36 a2 + 216 a3"""
    m = np.asarray(moves, np.uint16).reshape(-1, 4)
    return (m[:, 0] + 6 * m[:, 1] + 36 * m[:, 2] + 216 * m[:, 3]).astype(np.uint16)


class Stats(C.Structure):
    _fields_ = [("env_steps", C.c_uint64), ("episodes", C.c_uint64), ("wins", C.c_uint64 * 4),
                ("draws", C.c_uint64), ("truncated", C.c_uint64), ("sum_episode_len", C.c_uint64),
                ("invalid", C.c_uint64)]

    def as_dict(self):
        return {"env_steps": self.env_steps, "episodes": self.episodes, "wins": list(self.wins),
                "draws": self.draws, "truncated": self.truncated, "sum_episode_len": self.sum_episode_len,
                "invalid": self.invalid}

    def as_array(self):
        return np.array([self.env_steps, self.episodes, *self.wins, self.draws, self.truncated,
                         self.sum_episode_len, self.invalid], dtype=np.int64)


class PomError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("pom_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """Loads libpom_b200.so (built by __graft_entry__.build()).  No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
        L.pom_last_error.restype = C.c_char_p
        L.pom_batch_init.argtypes = [C.POINTER(vp), i32, u64, C.POINTER(InitDesc)]
        L.pom_batch_destroy.argtypes = [vp]
        L.pom_batch_sync.argtypes = [vp]
        L.pom_batch_upload.argtypes = [vp, u64, u64, vp, vp]
        L.pom_batch_download.argtypes = [vp, u64, u64, vp, vp]
        L.pom_batch_observe.argtypes = [vp, u64, u64, i32, i32, vp, vp]
        L.pom_batch_obs_stride.restype = u64
        L.pom_batch_obs_stride.argtypes = [vp]
        L.pom_batch_observe_planes.argtypes = [vp, vp, u32, i32]
        L.pom_batch_observe_planes_cropped.argtypes = [vp, vp, u32, i32]
        L.pom_obs_cropped_bytes.argtypes = [i32]
        L.pom_obs_cropped_bytes.restype = u32
        L.pom_device_copy.argtypes = [i32, vp, vp, u64]
        L.pom_batch_reset.argtypes = [vp]
        L.pom_batch_templates.argtypes = [vp, vp, vp]
        L.pom_batch_step.argtypes = [vp, vp, u32]
        L.pom_batch_step_host.argtypes = [vp, vp, vp, u32]
        L.pom_batch_step_host_async.argtypes = [vp, vp, vp, u32]
        L.pom_batch_rollout.argtypes = [vp, u32, u64, u32, u32]
        L.pom_batch_step_seq.argtypes = [vp, vp, u32, u32]
        L.pom_batch_policy_moves.argtypes = [vp, vp, u64, u32, u32]
        L.pom_batch_policy_moves_host.argtypes = [vp, vp, u64, u32, u32]
        L.pom_batch_policy_act.argtypes = [vp, u64, i32, i32, C.POINTER(C.c_int)]
        L.pom_batch_policy_reset.argtypes = [vp]
        L.pom_batch_policy_download.argtypes = [vp, u64, u64, vp]
        L.pom_batch_policy_upload.argtypes = [vp, u64, u64, vp]
        L.pom_batch_clone.argtypes = [vp, u64, vp, vp, u64]
        L.pom_batch_expand_step.argtypes = [vp, vp, vp, u64, u32, u32]
        L.pom_batch_spawn_flame.argtypes = [vp, u64, i32, i32, i32]
        L.pom_batch_apply.argtypes = [vp, u64, i32, i32, i32, i32]
        L.pom_make_board.argtypes = [i32, C.c_int32, vp, C.POINTER(C.c_int)]
        L.pom_batch_status.argtypes = [vp, u64, u64, vp]
        L.pom_batch_stats.argtypes = [vp, C.POINTER(Stats)]
        L.pom_batch_clear_stats.argtypes = [vp]
        L.pom_rng_moves.restype = u32
        L.pom_rng_moves.argtypes = [u64, u64, u32, u32]
        L.pom_batch_generate_moves.argtypes = [vp, vp, u64, u32, u32]
        L.pom_batch_size.restype = u64
        L.pom_batch_teams.argtypes = [vp]
        L.pom_batch_radio.argtypes = [vp]
        L.pom_batch_step_radio.argtypes = [vp, vp, vp, u32, vp, vp]
        L.pom_batch_radio_download.argtypes = [vp, u64, u64, vp]
        L.pom_batch_radio_upload.argtypes = [vp, u64, u64, vp]
        L.pom_batch_set_policy_view.argtypes = [vp, i32]
        L.pom_batch_get_policy_view.argtypes = [vp, C.POINTER(C.c_int)]
        L.pom_batch_size.argtypes = [vp]
        L.pom_batch_device.argtypes = [vp]
        for f in ("pom_batch_stream", "pom_batch_stats_device_ptr", "pom_batch_records_device_ptr"):
            getattr(L, f).restype = vp
            getattr(L, f).argtypes = [vp]
        L.pom_device_alloc.argtypes = [i32, u64, C.POINTER(vp)]
        L.pom_device_free.argtypes = [i32, vp]
        L.pom_host_alloc.argtypes = [u64, C.POINTER(vp)]
        L.pom_host_free.argtypes = [vp]
        L.pom_host_alloc_near.argtypes = [i32, u64, C.POINTER(vp)]
        L.pom_bind_thread_near.argtypes = [i32]
        L.pom_batch_step_compact.argtypes = [vp, vp, u32]
        L.pom_batch_step_observe.argtypes = [vp, vp, u32, vp, u32, i32]
        L.pom_batch_step_rewards.argtypes = [vp, vp, u32, vp, vp]
        L.pom_batch_event_record.argtypes = [vp, i32]
        L.pom_batch_event_elapsed_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.pom_batch_flush_l2.argtypes = [vp]
        L.pom_batch_launch_count.restype = u64
        L.pom_batch_launch_count.argtypes = [vp]
        _lib = L
    return _lib


def _ck(rc):
    if rc != 0:
        raise PomError(rc, lib().pom_last_error().decode())


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def device_count():
    return lib().pom_device_count()


class Batch:
    """One handle = one shard of envs on one GPU (pom_batch_* of include/pom_batch.h)."""

    def __init__(self, n_envs, device=0, env_offset=0, n_templates=1024, first_seed=0x1337,
                 host_templates=None, max_ticks=0, empty=False, teams=False, radio=False):
        self.h = C.c_void_p()
        d = InitDesc()
        d.env_offset = env_offset
        d.first_seed = first_seed
        d.max_ticks = max_ticks
        d.flags = (INIT_EMPTY if empty else 0) | (INIT_TEAMS if teams else 0) | (INIT_RADIO if radio else 0)
        self._keep = None
        if host_templates is not None:
            assert host_templates.dtype == STATE_DT
            self._keep = np.ascontiguousarray(host_templates)
            d.n_templates = self._keep.shape[0]
            d.host_templates = self._keep.ctypes.data
        else:
            d.n_templates = n_templates
            d.host_templates = None
        self.n_templates = d.n_templates
        self.n = n_envs
        self.device = device
        _ck(lib().pom_batch_init(C.byref(self.h), device, n_envs, C.byref(d)))

    def close(self):
        if self.h:
            lib().pom_batch_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self): _ck(lib().pom_batch_sync(self.h))

    def teams(self):
        """True if the handle plays the 2v2 team game (pom_batch_teams)"""
        r = lib().pom_batch_teams(self.h)
        _ck(min(r, 0))
        return r == 1

    def radio(self):
        """True if the handle has the team radio (pom_batch_radio; Batch(..., teams=True, radio=True))"""
        r = lib().pom_batch_radio(self.h)
        _ck(min(r, 0))
        return r == 1

    def records_compressed(self):
        """True if the record array lives in compressible device memory (pom_batch_records_compressed): a report, not a switch"""
        # looked up here, not bound in lib(), so that POM_B200_LIB can still load builds that predate it (A/B runs)
        f = lib().pom_batch_records_compressed
        f.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        v = C.c_int()
        _ck(f(self.h, C.byref(v)))
        return v.value == 1

    def radio_download(self, first=0, count=None):
        """[count, 4] uint8: every env's last message per agent, byte a = w0 | w1 << 3 (unpack_messages splits it)"""
        count = self.n - first if count is None else count
        m = np.zeros((count, 4), np.uint8)
        _ck(lib().pom_batch_radio_download(self.h, first, count, _p(m)))
        return m

    def radio_upload(self, msgs, first=0):
        """sets the last messages of envs first.. from [count, 4] bytes in the encoding of radio_download"""
        m = np.ascontiguousarray(msgs, dtype=np.uint8).reshape(-1, 4)
        _ck(lib().pom_batch_radio_upload(self.h, first, m.shape[0], _p(m)))

    def set_policy_view(self, view):
        """fog of war for the device SimpleAgent (pom_batch_set_policy_view): with view >= 0 every later call that runs it
        (policy_moves[_host], rollout with ROLL_SIMPLE, policy_act) plays it on what each agent sees through its square
        window of `view` cells; view < 0 (the default, -1) = the full state"""
        _ck(lib().pom_batch_set_policy_view(self.h, int(view)))

    def policy_view(self):
        """the view last set by set_policy_view (-1 if never set)"""
        v = C.c_int(0)
        _ck(lib().pom_batch_get_policy_view(self.h, C.byref(v)))
        return v.value
    def reset(self): _ck(lib().pom_batch_reset(self.h))

    def upload(self, states, status=None, first=0):
        assert states.dtype == STATE_DT and states.flags.c_contiguous
        _ck(lib().pom_batch_upload(self.h, first, states.shape[0], _p(states), _p(status)))

    def download(self, first=0, count=None, with_states=True):
        count = self.n - first if count is None else count
        S = np.zeros(count, STATE_DT) if with_states else None
        st = np.zeros(count, np.uint8)
        _ck(lib().pom_batch_download(self.h, first, count, _p(S), _p(st)))
        return S, st

    def observe(self, agent, view=4, first=0, count=None):
        """States as `agent` sees them through a (2*view+1)^2 window (fog of war)"""
        count = self.n - first if count is None else count
        S = np.zeros(count, STATE_DT)
        st = np.zeros(count, np.uint8)
        _ck(lib().pom_batch_observe(self.h, first, count, agent, view, _p(S), _p(st)))
        return S, st

    def observe_planes(self, agent_mask=15, view=4, obs_dev=None):
        """observation planes of the agents in agent_mask, computed and kept on the device; returns a host copy
        [n_agents, n_envs, 512] (and leaves obs_dev filled if the caller passed its own buffer)"""
        k = bin(agent_mask & 15).count("1")
        stride = int(lib().pom_batch_obs_stride(self.h))
        own = obs_dev is None
        if own:
            obs_dev = self.alloc(k * stride * OBS_BYTES)
        _ck(lib().pom_batch_observe_planes(self.h, obs_dev, agent_mask, view))
        self.sync()
        host = np.zeros((k, stride, OBS_BYTES), np.uint8)
        _ck(lib().pom_device_copy(self.device, _p(host), obs_dev, host.nbytes))
        if own:
            self.free(obs_dev)
        return host[:, :self.n]

    def observe_planes_cropped(self, agent_mask=15, view=4, obs_dev=None):
        """the cropped layout (pom_batch_observe_planes_cropped): returns a host copy [n_agents, n_envs, pom_obs_cropped_bytes(view)]"""
        k = bin(agent_mask & 15).count("1")
        stride = int(lib().pom_batch_obs_stride(self.h))
        rb = int(lib().pom_obs_cropped_bytes(view))
        own = obs_dev is None
        if own:
            obs_dev = self.alloc(k * stride * max(rb, 32))
        _ck(lib().pom_batch_observe_planes_cropped(self.h, obs_dev, agent_mask, view))
        self.sync()
        host = np.zeros((k, stride, rb), np.uint8)
        _ck(lib().pom_device_copy(self.device, _p(host), obs_dev, host.nbytes))
        if own:
            self.free(obs_dev)
        return host[:, :self.n]

    def templates(self):
        T = np.zeros(self.n_templates, STATE_DT)
        seeds = np.zeros(self.n_templates, np.int32)
        _ck(lib().pom_batch_templates(self.h, _p(T), _p(seeds)))
        return T, seeds

    def step(self, moves_dev, flags=0):
        _ck(lib().pom_batch_step(self.h, moves_dev, flags))

    def step_host(self, moves, status_out=None, flags=0):
        assert moves.dtype == np.uint8 and moves.size == 4 * self.n and moves.flags.c_contiguous
        _ck(lib().pom_batch_step_host(self.h, _p(moves), _p(status_out), flags))

    def step_observe(self, moves_dev, obs_dev, agent_mask=1, view=4, flags=0):
        """one tick + observation planes of the agents in agent_mask, one kernel (pom_batch_step_observe)"""
        _ck(lib().pom_batch_step_observe(self.h, moves_dev, flags, obs_dev, agent_mask, view))

    def compact_io(self, joint, done_bits=None, fin_env=None, fin_status=None, fin_count=None, obs_dev=None,
                   obs_agent_mask=0, obs_view=4):
        """a prepared pom_step_compact_io for step_compact_io (an actor loop reuses its buffers: build the struct once)"""
        def ptr(a):
            if a is None:
                return None
            return C.c_void_p(a) if isinstance(a, int) else _p(a)
        return StepCompactIO(ptr(joint), ptr(done_bits), ptr(fin_env), ptr(fin_status), ptr(fin_count),
                             0 if fin_env is None else (fin_env.size if hasattr(fin_env, "size") else self.n),
                             obs_dev, obs_agent_mask, obs_view)

    def step_compact_io(self, io, flags=0):
        _ck(lib().pom_batch_step_compact(self.h, C.byref(io), flags))

    def step_compact(self, joint, done_bits=None, fin_env=None, fin_status=None, fin_count=None, flags=0, obs_dev=None,
                     obs_agent_mask=0, obs_view=4):
        """one tick with compact I/O (pom_batch_step_compact): `joint` = n uint16 joint actions; outputs are optional.
        Arrays must live in pinned mapped memory (pinned_array) or be raw device pointers (int); enqueue only."""
        def ptr(a):
            if a is None:
                return None
            return C.c_void_p(a) if isinstance(a, int) else _p(a)
        io = StepCompactIO(ptr(joint), ptr(done_bits), ptr(fin_env), ptr(fin_status), ptr(fin_count),
                           0 if fin_env is None else (fin_env.size if hasattr(fin_env, "size") else self.n),
                           obs_dev, obs_agent_mask, obs_view)
        _ck(lib().pom_batch_step_compact(self.h, C.byref(io), flags))

    def step_rewards(self, moves_dev, rewards, status=None, flags=0):
        """one tick that also writes every env's four int8 rewards (pom_batch_step_rewards): `rewards` = n x 4 bytes,
        `status` = n status bytes (optional), as pom_batch_step_host reports them.  Arrays must live in pinned mapped memory
        (pinned_array) or be raw device pointers; enqueue only."""
        def ptr(a):
            return a if isinstance(a, (int, C.c_void_p)) else _p(a)
        _ck(lib().pom_batch_step_rewards(self.h, ptr(moves_dev), flags, ptr(rewards), ptr(status)))

    def step_radio(self, moves_dev, msgs, rewards=None, status=None, flags=0):
        """one tick of step_rewards with the team radio (pom_batch_step_radio): `msgs` = n x 4 message bytes (pack_messages),
        `rewards` (n x 4 int8) and `status` (n bytes) optional.  Arrays must live in pinned mapped memory (pinned_array) or be
        raw device pointers; enqueue only."""
        def ptr(a):
            return a if isinstance(a, (int, C.c_void_p)) or a is None else _p(a)
        _ck(lib().pom_batch_step_radio(self.h, ptr(moves_dev), ptr(msgs), flags, ptr(rewards), ptr(status)))

    def step_seq(self, moves_dev, ticks, flags=0):
        """`ticks` ticks in one launch with the caller's moves (device pointer, ticks x n x 4 bytes, tick-major)"""
        _ck(lib().pom_batch_step_seq(self.h, moves_dev, ticks, flags))

    def step_host_async(self, moves, status_out=None, flags=0):
        """pinned buffers only; results are valid after sync()"""
        assert moves.dtype == np.uint8 and moves.size == 4 * self.n and moves.flags.c_contiguous
        _ck(lib().pom_batch_step_host_async(self.h, _p(moves), _p(status_out), flags))

    def rollout(self, ticks, seed, tick0=0, flags=0):
        _ck(lib().pom_batch_rollout(self.h, ticks, seed, tick0, flags))

    def policy_moves(self, moves_dev, seed, tick, agent_mask=15):
        _ck(lib().pom_batch_policy_moves(self.h, moves_dev, seed, tick, agent_mask))

    def policy_moves_host(self, moves, seed, tick, agent_mask=15):
        assert moves.dtype == np.uint8 and moves.size == 4 * self.n and moves.flags.c_contiguous
        _ck(lib().pom_batch_policy_moves_host(self.h, _p(moves), seed, tick, agent_mask))

    def policy_act(self, env, agent, draw):
        m = C.c_int(0)
        _ck(lib().pom_batch_policy_act(self.h, env, agent, draw, C.byref(m)))
        return m.value

    def policy_reset(self): _ck(lib().pom_batch_policy_reset(self.h))

    def policy_download(self, first=0, count=None):
        count = self.n - first if count is None else count
        A = np.zeros((count, 4), SIMPLE_DT)
        _ck(lib().pom_batch_policy_download(self.h, first, count, _p(A)))
        return A

    def policy_upload(self, A, first=0):
        assert A.dtype == SIMPLE_DT and A.flags.c_contiguous and A.shape[1] == 4
        _ck(lib().pom_batch_policy_upload(self.h, first, A.shape[0], _p(A)))

    def clone_from(self, src, src_idx, first_dst=0):
        idx = np.ascontiguousarray(src_idx, dtype=np.uint32)
        _ck(lib().pom_batch_clone(self.h, first_dst, src.h, _p(idx), idx.shape[0]))

    def expand_step_from(self, src, root_idx, fanout=1296, flags=0):
        idx = np.ascontiguousarray(root_idx, dtype=np.uint32)
        _ck(lib().pom_batch_expand_step(self.h, src.h, _p(idx), idx.shape[0], fanout, flags))

    def spawn_flame(self, env, x, y, strength):
        _ck(lib().pom_batch_spawn_flame(self.h, env, x, y, strength))

    def apply(self, env, op, a0=0, a1=0, a2=0):
        _ck(lib().pom_batch_apply(self.h, env, op, a0, a1, a2))

    def status(self, first=0, count=None):
        return self.download(first, count, with_states=False)[1]

    def stats(self):
        s = Stats()
        _ck(lib().pom_batch_stats(self.h, C.byref(s)))
        return s

    def clear_stats(self): _ck(lib().pom_batch_clear_stats(self.h))

    def alloc(self, nbytes):
        p = C.c_void_p()
        _ck(lib().pom_device_alloc(self.device, nbytes, C.byref(p)))
        return p

    def free(self, p): _ck(lib().pom_device_free(self.device, p))

    def generate_moves(self, moves_dev, seed, tick, n_actions=6):
        _ck(lib().pom_batch_generate_moves(self.h, moves_dev, seed, tick, n_actions))

    def event(self, which): _ck(lib().pom_batch_event_record(self.h, which))

    def elapsed_ms(self):
        ms = C.c_float(0)
        _ck(lib().pom_batch_event_elapsed_ms(self.h, C.byref(ms)))
        return ms.value

    def flush_l2(self): _ck(lib().pom_batch_flush_l2(self.h))
    def launch_count(self): return int(lib().pom_batch_launch_count(self.h))
    def stats_device_ptr(self): return lib().pom_batch_stats_device_ptr(self.h)
    def stream(self): return lib().pom_batch_stream(self.h)


def make_board(seed, device=0):
    """InitBoardItems(state, seed) generated on the device; returns (state, dirty)."""
    s = np.zeros(1, STATE_DT)
    d = C.c_int(0)
    _ck(lib().pom_make_board(device, seed, _p(s), C.byref(d)))
    return s, d.value


def bind_thread_near(device):
    """pins the calling thread to the CPUs next to `device` (pom_bind_thread_near)"""
    _ck(lib().pom_bind_thread_near(device))


def pinned_array(shape, dtype, near_device=None):
    """numpy array backed by pinned host memory (pom_host_alloc, or pom_host_alloc_near when near_device is given: pages
    on the GPU's NUMA node); keep the returned owner alive."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    if near_device is None:
        _ck(lib().pom_host_alloc(n, C.byref(p)))
    else:
        _ck(lib().pom_host_alloc_near(near_device, n, C.byref(p)))
    buf = (C.c_uint8 * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    return arr, p


def pinned_free(p):
    _ck(lib().pom_host_free(p))


def rng_moves(seed, env0, n, tick, n_actions=6):
    """Host evaluation of the shared stateless action source (pom_rng_moves)."""
    out = np.zeros(n, np.uint32)
    f = lib().pom_rng_moves
    for e in range(n):
        out[e] = f(seed, env0 + e, tick, n_actions)
    return out.view(np.uint8).reshape(n, 4)
