"""TEST INFRASTRUCTURE: ctypes wrapper around ``oracle/_build/liblob_oracle.so`` (see lob_oracle.c).

One ``Oracle`` object == one environment (one reference ``HistoricalOrderbookEnvironment`` /
``OrderbookSimulator`` / ``Exchange``).
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from rl4mm_b200 import abi
from rl4mm_b200.packing import PackedStream

_HERE = Path(__file__).resolve().parent
_LIB = None


def build(force: bool = False) -> Path:
    so = _HERE / "_build" / "liblob_oracle.so"
    src = [_HERE / "lob_oracle.c", _HERE / "lob_oracle.h", _HERE.parent / "include" / "lobsim.h"]
    stale = lambda: force or not so.exists() or any(s.stat().st_mtime > so.stat().st_mtime for s in src)   # noqa: E731
    if stale():
        import fcntl

        (_HERE / "_build").mkdir(exist_ok=True)
        with open(_HERE / "_build" / ".lock", "w") as lock:        # pytest-xdist workers: one builds, the others wait and re-check
            fcntl.flock(lock, fcntl.LOCK_EX)
            if stale():
                subprocess.run(["make", "-C", str(_HERE), "-s", "-B"], check=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(str(build()))
        L.lo_create.restype = C.c_void_p
        L.lo_create.argtypes = [C.POINTER(abi.Cfg)]
        L.lo_destroy.argtypes = [C.c_void_p]
        L.lo_set_stream.argtypes = [C.c_void_p, C.POINTER(abi.Stream)]
        L.lo_reset_book.argtypes = [C.c_void_p, C.c_int]
        L.lo_reset.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.lo_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lo_replay.argtypes = [C.c_void_p, C.c_int]
        L.lo_forward_step.argtypes = [C.c_void_p, C.c_int]
        L.lo_set_book.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.lo_peaks.argtypes = [C.c_void_p, C.c_void_p]
        L.lo_rollout.argtypes = [C.c_void_p, C.c_int, C.POINTER(abi.Agent), C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
        L.lo_rollout_info.argtypes = [C.c_void_p, C.c_int, C.POINTER(abi.Agent), C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
        L.lo_agent_action.argtypes = [C.POINTER(abi.Agent), C.c_void_p, C.c_void_p]
        L.lo_philox4x32_10.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.lo_random_action.argtypes = [C.POINTER(abi.Agent), C.c_int32, C.c_int64, C.c_void_p]
        L.lo_set_env_index.argtypes = [C.c_void_p, C.c_int32]
        L.lo_action_to_ladders.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lo_process_order.argtypes = [C.c_void_p, C.POINTER(abi.Order), C.POINTER(C.c_uint32)]
        L.lo_clear_fills.argtypes = [C.c_void_p]
        L.lo_get_fills.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.lo_dump_book.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.lo_dump_agent_orders.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.lo_get_state.argtypes = [C.c_void_p, C.c_void_p]
        L.lo_obs_dim.argtypes = [C.POINTER(abi.Cfg)]
        L.lo_action_dim.argtypes = [C.POINTER(abi.Cfg)]
        _LIB = L
    return _LIB


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self, cfg: abi.Cfg, stream: PackedStream | None = None, env_index: int = 0):
        self.cfg = cfg
        self._h = lib().lo_create(C.byref(cfg))
        lib().lo_set_env_index(self._h, env_index)        # part of the RandomAgent stream key
        self._keep = None
        self.obs_dim = lib().lo_obs_dim(C.byref(cfg))
        self.action_dim = lib().lo_action_dim(C.byref(cfg))
        if stream is not None:
            self.set_stream(stream)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().lo_destroy(self._h)
            self._h = None

    def set_stream(self, s: PackedStream):
        assert s.n_levels == self.cfg.n_levels and s.step_us == self.cfg.step_us
        st = abi.Stream(s.msgs.ctypes.data, s.n_msgs, s.step_off.ctypes.data, s.n_grid_steps, s.snapshots.ctypes.data,
                        s.snap_valid.ctypes.data, s.n_seconds, 0, s.t0_us)
        self._keep = (s, st)
        lib().lo_set_stream(self._h, C.byref(st))

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f"oracle call failed: {rc}")

    def reset_book(self, start_step: int):
        self._check(lib().lo_reset_book(self._h, int(start_step)))

    def reset(self, episode_start_step: int) -> np.ndarray:
        obs = np.zeros(self.obs_dim)
        self._check(lib().lo_reset(self._h, int(episode_start_step), _ptr(obs)))
        return obs

    def step(self, action):
        a = np.ascontiguousarray(action, dtype=np.float64)
        assert a.shape == (self.action_dim,)
        obs = np.zeros(self.obs_dim)
        r = np.zeros(1)
        d = np.zeros(1, np.uint8)
        self._check(lib().lo_step(self._h, _ptr(a), _ptr(obs), _ptr(r), _ptr(d)))
        return obs, float(r[0]), bool(d[0])

    def replay(self, n_steps: int):
        self._check(lib().lo_replay(self._h, int(n_steps)))

    def forward_step(self, n_steps: int):
        """One OrderbookSimulator.forward_step over n_steps grid steps: the resync condition is evaluated once, at the end."""
        self._check(lib().lo_forward_step(self._h, int(n_steps)))

    def set_book(self, buy: np.ndarray, sell: np.ndarray):
        """Replace the books by L3 entries in the dump_book format (agent entries also form the internal book)."""
        buy = np.ascontiguousarray(buy, dtype=abi.BOOK_ENTRY_DTYPE)
        sell = np.ascontiguousarray(sell, dtype=abi.BOOK_ENTRY_DTYPE)
        self._check(lib().lo_set_book(self._h, _ptr(buy), len(buy), _ptr(sell), len(sell)))

    def peaks(self) -> dict:
        """Capacity high-water marks since the last reset_book / reset / set_book, counted like the device book: price levels,
        resting orders (snapshot aggregates included) and agent orders per side [buy, sell], and the most fills of one call."""
        out = np.zeros(7, np.int32)
        lib().lo_peaks(self._h, _ptr(out))
        return dict(levels=(int(out[0]), int(out[1])), orders=(int(out[2]), int(out[3])), agents=(int(out[4]), int(out[5])),
                    fills=int(out[6]))

    def rollout(self, T: int, agent: abi.Agent, actions=None, want_info=False):
        obs = np.zeros((T, self.obs_dim))
        act = np.zeros((T, self.action_dim)) if actions is None else np.ascontiguousarray(actions, np.float64)
        rew = np.zeros(T)
        done = np.zeros(T, np.uint8)
        if want_info:
            info = np.zeros((T, abi.INFO_DIM))
            self._check(lib().lo_rollout_info(self._h, T, C.byref(agent), _ptr(obs), _ptr(act), _ptr(rew), _ptr(done), _ptr(info)))
            return obs, act, rew, done, info
        self._check(lib().lo_rollout(self._h, T, C.byref(agent), _ptr(obs), _ptr(act), _ptr(rew), _ptr(done)))
        return obs, act, rew, done

    def action_to_ladders(self, action):
        a = np.ascontiguousarray(action, np.float64)
        q = self.cfg.max_quote_level - self.cfg.min_quote_level
        buy, sell = np.zeros(q, np.int64), np.zeros(q, np.int64)
        lib().lo_action_to_ladders(self._h, _ptr(a), _ptr(buy), _ptr(sell))
        return buy, sell

    def process_order(self, type, direction, price, volume, is_external, ref) -> int:
        o = abi.Order(0, type, direction, price, volume, int(is_external), ref, 0)
        out = C.c_uint32(0)
        self._check(lib().lo_process_order(self._h, C.byref(o), C.byref(out)))
        return out.value

    def clear_fills(self):
        lib().lo_clear_fills(self._h)

    def fills(self) -> np.ndarray:
        n = lib().lo_get_fills(self._h, None, 0)
        out = np.zeros(n, abi.FILL_DTYPE)
        lib().lo_get_fills(self._h, _ptr(out), n)
        return out

    def dump_book(self, side: int) -> np.ndarray:
        n = lib().lo_dump_book(self._h, side, None, 0)
        out = np.zeros(n, abi.BOOK_ENTRY_DTYPE)
        lib().lo_dump_book(self._h, side, _ptr(out), n)
        return out

    def dump_agent_orders(self, side: int) -> np.ndarray:
        n = lib().lo_dump_agent_orders(self._h, side, None, 0)
        out = np.zeros(n, abi.BOOK_ENTRY_DTYPE)
        lib().lo_dump_agent_orders(self._h, side, _ptr(out), n)
        return out

    def state(self) -> np.ndarray:
        st = np.zeros(1, abi.ENV_STATE_DTYPE)
        lib().lo_get_state(self._h, _ptr(st))
        return st[0]


def philox4x32_10(ctr, key) -> list:
    c = np.array(ctr, np.uint32)
    lib().lo_philox4x32_10(_ptr(c), int(key[0]), int(key[1]))
    return [int(x) for x in c]


def random_action(agent: abi.Agent, env_index: int, now_step: int) -> np.ndarray:
    a = np.zeros(5)
    lib().lo_random_action(C.byref(agent), env_index, now_step, _ptr(a))
    return a


def agent_action(agent: abi.Agent, obs) -> np.ndarray:
    o = np.ascontiguousarray(obs, np.float64)
    a = np.zeros(5)
    lib().lo_agent_action(C.byref(agent), _ptr(o), _ptr(a))
    return a
