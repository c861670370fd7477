"""Batched device handle: N environments (books) on one GPU, driven through the C ABI.

PyTorch is used for device memory, streams and (elsewhere) torch.distributed only; all compute is in
``liblobsim.so``.  Tensors returned by this class are torch CUDA tensors (float64 unless stated otherwise).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import abi
from ._lib import LobsimError, check, lib, np_ptr
from .packing import PackedStream


def _dptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class DeviceStream:
    """A PackedStream resident in HBM (the device-side replacement of the reference's Postgres tables)."""

    def __init__(self, packed: PackedStream, device: torch.device):
        packed.validate()
        self.packed = packed
        self.msgs = torch.from_numpy(packed.msgs.view(np.uint8).reshape(-1, 16).copy()).to(device)
        if self.msgs.numel() == 0:
            self.msgs = torch.zeros((1, 16), dtype=torch.uint8, device=device)
        self.step_off = torch.from_numpy(packed.step_off.view(np.int32).copy()).to(device)  # uint32 bits
        self.snapshots = torch.from_numpy(packed.snapshots.copy()).to(device)
        self.snap_valid = torch.from_numpy(packed.snap_valid.copy()).to(device)
        self.struct = abi.Stream(self.msgs.data_ptr(), packed.n_msgs, self.step_off.data_ptr(), packed.n_grid_steps,
                                 self.snapshots.data_ptr(), self.snap_valid.data_ptr(), packed.n_seconds, 0,
                                 packed.t0_us)


class LobSim:
    def __init__(self, cfg: abi.Cfg, device: int = 0):
        if not torch.cuda.is_available():
            raise LobsimError("no CUDA device: the lobsim hot path has no CPU fallback")
        self.cfg = cfg
        self.device_index = device
        self.device = torch.device("cuda", device)
        self.n_envs = cfg.n_envs
        self.obs_dim = abi.obs_dim(cfg)
        self.action_dim = abi.action_dim(cfg)
        h = C.c_void_p()
        check(lib().lobsim_create(C.byref(cfg), device, C.byref(h)))
        self._h = h
        self._streams: dict[int, DeviceStream] = {}

    def close(self):
        if getattr(self, "_h", None):
            lib().lobsim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- streams -----------------------------------------------------------------------------------------------
    def load_stream(self, stream_id: int, packed: PackedStream) -> DeviceStream:
        if packed.n_levels != self.cfg.n_levels or packed.step_us != self.cfg.step_us:
            raise ValueError("stream n_levels / step_us do not match the configuration")
        ds = DeviceStream(packed, self.device)
        check(lib().lobsim_load_stream(self._h, stream_id, C.byref(ds.struct)))
        self._streams[stream_id] = ds
        return ds

    def _i32(self, x, n) -> torch.Tensor:
        if isinstance(x, torch.Tensor):
            t = x.to(device=self.device, dtype=torch.int32).contiguous()
        else:
            t = torch.as_tensor(np.broadcast_to(np.asarray(x, dtype=np.int32), (n,)).copy(), device=self.device)
        assert t.shape == (n,)
        return t

    def _stream_arg(self, stream):
        return C.c_void_p(stream.cuda_stream) if stream is not None else C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- reset / step / rollout / replay -------------------------------------------------------------------------
    def reset(self, stream_ids, episode_start_steps, env_ids=None, stream=None) -> torch.Tensor:
        n = self.n_envs if env_ids is None else len(env_ids)
        ids = None if env_ids is None else self._i32(env_ids, n)
        sid, st = self._i32(stream_ids, n), self._i32(episode_start_steps, n)
        obs = torch.empty((n, self.obs_dim), dtype=torch.float64, device=self.device)
        check(lib().lobsim_reset(self._h, _dptr(ids), n, _dptr(sid), _dptr(st), _dptr(obs), self._stream_arg(stream)))
        return obs

    def reset_book(self, stream_ids, start_steps, env_ids=None, stream=None) -> None:
        n = self.n_envs if env_ids is None else len(env_ids)
        ids = None if env_ids is None else self._i32(env_ids, n)
        sid, st = self._i32(stream_ids, n), self._i32(start_steps, n)
        check(lib().lobsim_reset_book(self._h, _dptr(ids), n, _dptr(sid), _dptr(st), self._stream_arg(stream)))

    def step(self, actions: torch.Tensor, stream=None):
        a = actions.to(device=self.device, dtype=torch.float64).contiguous()
        assert a.shape == (self.n_envs, self.action_dim), a.shape
        obs = torch.empty((self.n_envs, self.obs_dim), dtype=torch.float64, device=self.device)
        rew = torch.empty(self.n_envs, dtype=torch.float64, device=self.device)
        done = torch.empty(self.n_envs, dtype=torch.uint8, device=self.device)
        check(lib().lobsim_step(self._h, _dptr(a), _dptr(obs), _dptr(rew), _dptr(done), self._stream_arg(stream)))
        return obs, rew, done

    def step_host(self, actions: np.ndarray, obs: np.ndarray, rew: np.ndarray, done: np.ndarray) -> None:
        """HOST buffers in / out (pinned recommended); the library does the H2D / D2H copies."""
        assert actions.dtype == np.float64 and actions.shape == (self.n_envs, self.action_dim)
        check(lib().lobsim_step_host(self._h, np_ptr(actions), np_ptr(obs), np_ptr(rew), np_ptr(done)))

    def rollout(self, T: int, agent: abi.Agent, actions: Optional[torch.Tensor] = None, want_obs=True, stream=None,
                want_info=False):
        """Fused T-step rollout; with ``want_info`` a fifth tensor info [T, N, abi.INFO_DIM] is returned as well.
        ``agent`` may be a sequence of n_envs built-in agents (one per env: parameter sweeps)."""
        N = self.n_envs
        if not isinstance(agent, abi.Agent):
            agents = (abi.Agent * N)(*agent)
            assert len(agent) == N, "one agent per env"
            obs = torch.empty((T, N, self.obs_dim), dtype=torch.float64, device=self.device) if want_obs else None
            act = torch.zeros((T, N, self.action_dim), dtype=torch.float64, device=self.device)
            rew = torch.zeros((T, N), dtype=torch.float64, device=self.device)
            done = torch.zeros((T, N), dtype=torch.uint8, device=self.device)
            info = torch.empty((T, N, abi.INFO_DIM), dtype=torch.float64, device=self.device) if want_info else None
            check(lib().lobsim_rollout_agents(self._h, T, C.cast(agents, C.c_void_p), _dptr(obs), _dptr(act), _dptr(rew), _dptr(done),
                                              _dptr(info), self._stream_arg(stream)))
            return (obs, act, rew, done, info) if want_info else (obs, act, rew, done)
        obs = torch.empty((T, N, self.obs_dim), dtype=torch.float64, device=self.device) if want_obs else None
        if agent.kind == abi.AGENT_EXTERNAL:
            act = actions.to(device=self.device, dtype=torch.float64).contiguous()
            assert act.shape == (T, N, self.action_dim)
        else:
            act = torch.zeros((T, N, self.action_dim), dtype=torch.float64, device=self.device)
        rew = torch.zeros((T, N), dtype=torch.float64, device=self.device)
        done = torch.zeros((T, N), dtype=torch.uint8, device=self.device)
        if want_info:
            info = torch.empty((T, N, abi.INFO_DIM), dtype=torch.float64, device=self.device)
            check(lib().lobsim_rollout_info(self._h, T, C.byref(agent), _dptr(obs), _dptr(act), _dptr(rew), _dptr(done),
                                            _dptr(info), self._stream_arg(stream)))
            return obs, act, rew, done, info
        check(lib().lobsim_rollout(self._h, T, C.byref(agent), _dptr(obs), _dptr(act), _dptr(rew), _dptr(done),
                                   self._stream_arg(stream)))
        return obs, act, rew, done

    def replay(self, n_steps: int, stream=None) -> None:
        check(lib().lobsim_replay(self._h, int(n_steps), self._stream_arg(stream)))

    def forward_step(self, n_steps: int, stream=None) -> None:
        """One OrderbookSimulator.forward_step over ``n_steps`` grid steps (resync evaluated once, at the end)."""
        check(lib().lobsim_forward_step(self._h, int(n_steps), self._stream_arg(stream)))

    def set_book(self, env: int, buy: np.ndarray, sell: np.ndarray) -> None:
        buy = np.ascontiguousarray(buy, dtype=abi.BOOK_ENTRY_DTYPE)
        sell = np.ascontiguousarray(sell, dtype=abi.BOOK_ENTRY_DTYPE)
        check(lib().lobsim_set_book(self._h, env, np_ptr(buy), len(buy), np_ptr(sell), len(sell)))

    def replay_host(self, stream_id: int, msgs_host: np.ndarray, first_msg: int, n_steps: int,
                    state_out: Optional[np.ndarray] = None) -> None:
        """Upload ``msgs_host`` (a slice of the stream starting at message ``first_msg``) and replay ``n_steps``."""
        assert msgs_host.dtype == abi.MSG_DTYPE and msgs_host.flags.c_contiguous
        if state_out is not None:
            assert state_out.dtype == abi.ENV_STATE_DTYPE and state_out.shape == (self.n_envs,)
        check(lib().lobsim_replay_host(self._h, stream_id, np_ptr(msgs_host), first_msg, len(msgs_host), int(n_steps),
                                       np_ptr(state_out) if state_out is not None else None))

    # ---- Exchange-level entry point and inspection ---------------------------------------------------------------
    def process_orders(self, orders: np.ndarray, max_fills: int = 4096):
        orders = np.ascontiguousarray(orders, dtype=abi.ORDER_DTYPE)
        fills = np.zeros(max_fills, abi.FILL_DTYPE)
        refs = np.zeros(len(orders), np.uint32)
        nf = C.c_int32(0)
        torch.cuda.synchronize(self.device)
        check(lib().lobsim_process_orders(self._h, np_ptr(orders), len(orders), np_ptr(fills), max_fills, C.byref(nf),
                                          np_ptr(refs)))
        return fills[: nf.value], refs

    def dump_book(self, env: int, side: int) -> np.ndarray:
        torch.cuda.synchronize(self.device)
        n = lib().lobsim_dump_book(self._h, env, side, None, 0)
        if n < 0:
            check(n)
        out = np.zeros(n, abi.BOOK_ENTRY_DTYPE)
        lib().lobsim_dump_book(self._h, env, side, np_ptr(out), n)
        return out

    def dump_agent_orders(self, env: int, side: int) -> np.ndarray:
        torch.cuda.synchronize(self.device)
        n = lib().lobsim_dump_agent_orders(self._h, env, side, None, 0)
        if n < 0:
            check(n)
        out = np.zeros(n, abi.BOOK_ENTRY_DTYPE)
        lib().lobsim_dump_agent_orders(self._h, env, side, np_ptr(out), n)
        return out

    def book_depth(self, depth: int, orders: bool = False, agent: bool = False, out=None, stream=None):
        """L2 depth of every env's central book, read on the device in one launch (lobsim_get_depth_dev): the L2
        projection of ``dump_book`` (rl4mm/extras/orderbook_comparison.py:6-19) for all envs at once.

        Returns torch CUDA tensors ``price`` int32 [N, 2, depth] (side 0 = buy, level 0 = best; absent levels
        ``abi.NO_PRICE``) and ``volume`` int64 [N, 2, depth] (agent orders and snapshot aggregates included), then
        ``orders`` int32 [N, 2, depth] (resting orders per level) if ``orders``, then ``agent_volume`` int64 [N, 2, depth]
        (the agent's own part of ``volume``, HOE.py:324) if ``agent``.  ``out``: a tuple of preallocated tensors in that
        order, filled and returned instead (for CUDA graph capture).  No host synchronisation; the books are read in
        whatever form they are in and left unchanged."""
        depth = int(depth)
        if not 1 <= depth <= self.cfg.max_levels_per_side:
            raise LobsimError(f"depth must be in [1, max_levels_per_side = {self.cfg.max_levels_per_side}], got {depth}")
        want = [torch.int32, torch.int64] + ([torch.int32] if orders else []) + ([torch.int64] if agent else [])
        shape = (self.n_envs, 2, depth)
        if out is None:
            out = tuple(torch.empty(shape, dtype=dt, device=self.device) for dt in want)
        else:
            out = tuple(out)
            if len(out) != len(want):
                raise ValueError(f"out: expected {len(want)} tensors (price, volume[, orders][, agent_volume])")
            for t, dt in zip(out, want):
                if t.dtype != dt or tuple(t.shape) != shape or t.device != self.device or not t.is_contiguous():
                    raise ValueError(f"out: expected contiguous {dt} tensors of shape {shape} on {self.device}")
        price, volume = out[0], out[1]
        n_orders = out[2] if orders else None
        agent_volume = out[-1] if agent else None
        check(lib().lobsim_get_depth_dev(self._h, depth, _dptr(price), _dptr(volume), _dptr(n_orders), _dptr(agent_volume),
                                         self._stream_arg(stream)))
        return out

    def agent_orders(self, max_orders: Optional[int] = None, queue: bool = True, out=None, stream=None):
        """The agent's resting orders of every env and their queue positions, read on the device in one launch
        (lobsim_get_agent_orders_dev): ``dump_agent_orders`` for all envs at once, plus where each order stands in the central
        book (Exchange._find_queue_position, Exchange.py:196-217).

        Returns torch CUDA tensors ``count`` int32 [N, 2] (agent orders per side, also beyond ``max_orders``, which
        defaults to ``cfg.max_agent_orders``), then ``price``, ``volume`` and ``id`` (the internal agent id) int32
        [N, 2, max_orders]: side 0 = buy, slots in ascending id, unused slots ``abi.NO_PRICE`` / 0 / 0.  With ``queue``
        also ``level`` int32 (0 = the best central level of the side, -1 for an unused slot), ``ahead_orders`` int32 and
        ``ahead_volume`` int64 (the resting orders in front of the order in the FIFO at its price, and their volume).
        ``out``: a tuple of preallocated tensors in that order, filled and returned instead (for CUDA graph capture).  No
        host synchronisation; the books are read in whatever form they are in and left unchanged."""
        A = self.cfg.max_agent_orders if max_orders is None else int(max_orders)
        if not 1 <= A <= self.cfg.max_agent_orders:
            raise LobsimError(f"max_orders must be in [1, max_agent_orders = {self.cfg.max_agent_orders}], got {A}")
        N = self.n_envs
        want = [((N, 2), torch.int32)] + [((N, 2, A), torch.int32)] * 3
        if queue:
            want += [((N, 2, A), torch.int32)] * 2 + [((N, 2, A), torch.int64)]
        if out is None:
            out = tuple(torch.empty(shape, dtype=dt, device=self.device) for shape, dt in want)
        else:
            out = tuple(out)
            if len(out) != len(want):
                raise ValueError(f"out: expected {len(want)} tensors (count, price, volume, id"
                                 + (", level, ahead_orders, ahead_volume)" if queue else ")"))
            for t, (shape, dt) in zip(out, want):
                if t.dtype != dt or tuple(t.shape) != shape or t.device != self.device or not t.is_contiguous():
                    raise ValueError(f"out: expected a contiguous {dt} tensor of shape {shape} on {self.device}")
        q = out[4:] if queue else (None, None, None)
        check(lib().lobsim_get_agent_orders_dev(self._h, A, *(_dptr(t) for t in out[:4]), *(_dptr(t) for t in q),
                                                self._stream_arg(stream)))
        return out

    def state(self, first: int = 0, n: Optional[int] = None) -> np.ndarray:
        n = self.n_envs - first if n is None else n
        out = np.zeros(n, abi.ENV_STATE_DTYPE)
        torch.cuda.synchronize(self.device)
        check(lib().lobsim_get_state(self._h, first, n, np_ptr(out)))
        return out

    def state_dev(self, stream=None) -> torch.Tensor:
        out = torch.empty((self.n_envs, abi.ENV_STATE_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        check(lib().lobsim_get_state_dev(self._h, _dptr(out), self._stream_arg(stream)))
        return out

    def fills(self, env: int) -> np.ndarray:
        torch.cuda.synchronize(self.device)
        cap = max(1, self.cfg.fill_log_capacity)
        out = np.zeros(cap, abi.FILL_DTYPE)
        n = C.c_int32(0)
        check(lib().lobsim_get_fills(self._h, env, np_ptr(out), cap, C.byref(n)))
        return out[: min(n.value, cap)]

    def errors(self) -> np.ndarray:
        """Per-env error bits (lobsim_errors: one strided device-to-host copy of the header words, no state summary)."""
        out = np.zeros(self.n_envs, np.uint32)
        torch.cuda.synchronize(self.device)
        check(lib().lobsim_errors(self._h, np_ptr(out)))
        return out

    @property
    def kernel_path(self) -> str:
        """"fast": the straight-line static-layout kernels serve this handle; "general": the runtime-layout kernel
        (capacities without a compiled layout, csrc/layouts.h, or LOBSIM_FORCE_GENERAL=1); "deep": capacities whose book exceeds
        the shared memory of an SM -- the general kernel works on the blobs in place in HBM (no capacity cliff, slower)."""
        return {abi.PATH_FAST: "fast", abi.PATH_DEEP: "deep"}.get(lib().lobsim_kernel_path(self._h), "general")

    @property
    def launch_count(self) -> int:
        return int(lib().lobsim_launch_count(self._h))

    @property
    def state_bytes(self) -> int:
        return int(lib().lobsim_state_bytes(C.byref(self.cfg)))
