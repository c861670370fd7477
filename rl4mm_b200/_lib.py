"""ctypes binding of ``rl4mm_b200/_native/liblobsim.so`` (the C ABI of include/lobsim.h).

There is NO CPU fallback: if the shared library is missing or no CUDA device is present, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import abi

_NATIVE = Path(__file__).resolve().parent / "_native" / "liblobsim.so"
_LIB = None


class LobsimError(RuntimeError):
    pass


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    import os

    native = Path(os.environ["LOBSIM_NATIVE_LIB"]) if os.environ.get("LOBSIM_NATIVE_LIB") else _NATIVE   # A/B builds (tools/)
    if not native.exists():
        raise LobsimError(
            f"{native} is missing: build the CUDA extension first (python -m rl4mm_b200.build, or "
            "__graft_entry__.build()).  The lobsim hot path has no CPU fallback."
        )
    L = C.CDLL(str(native))
    vp, i32, u32, i64, u64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_int64, C.c_uint64
    sig = {
        "lobsim_last_error": (C.c_char_p, []),
        "lobsim_abi_version": (C.c_int, []),
        "lobsim_state_bytes": (i64, [C.POINTER(abi.Cfg)]),
        "lobsim_create": (C.c_int, [C.POINTER(abi.Cfg), C.c_int, C.POINTER(vp)]),
        "lobsim_destroy": (C.c_int, [vp]),
        "lobsim_load_stream": (C.c_int, [vp, C.c_int, C.POINTER(abi.Stream)]),
        "lobsim_reset": (C.c_int, [vp, vp, i32, vp, vp, vp, vp]),
        "lobsim_step": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "lobsim_step_host": (C.c_int, [vp, vp, vp, vp, vp]),
        "lobsim_rollout": (C.c_int, [vp, i32, C.POINTER(abi.Agent), vp, vp, vp, vp, vp]),
        "lobsim_rollout_info": (C.c_int, [vp, i32, C.POINTER(abi.Agent), vp, vp, vp, vp, vp, vp]),
        "lobsim_rollout_agents": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp]),
        "lobsim_replay": (C.c_int, [vp, i32, vp]),
        "lobsim_forward_step": (C.c_int, [vp, i32, vp]),
        "lobsim_set_book": (C.c_int, [vp, i32, vp, i32, vp, i32]),
        "lobsim_replay_host": (C.c_int, [vp, C.c_int, vp, u64, u64, i32, vp]),
        "lobsim_reset_book": (C.c_int, [vp, vp, i32, vp, vp, vp]),
        "lobsim_process_orders": (C.c_int, [vp, vp, i32, vp, i32, C.POINTER(i32), vp]),
        "lobsim_submit_orders_dev": (C.c_int, [vp, i32, vp, vp, vp, i32, vp, vp, vp]),
        "lobsim_dump_book": (C.c_int, [vp, i32, i32, vp, i32]),
        "lobsim_dump_agent_orders": (C.c_int, [vp, i32, i32, vp, i32]),
        "lobsim_get_depth_dev": (C.c_int, [vp, i32, vp, vp, vp, vp, vp]),
        "lobsim_get_agent_orders_dev": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
        "lobsim_get_book_dev": (C.c_int, [vp, i32, vp, vp, vp]),
        "lobsim_set_book_dev": (C.c_int, [vp, i32, vp, vp, vp, vp]),
        "lobsim_get_state": (C.c_int, [vp, i32, i32, vp]),
        "lobsim_get_state_dev": (C.c_int, [vp, vp, vp]),
        "lobsim_get_fills": (C.c_int, [vp, i32, vp, i32, C.POINTER(i32)]),
        "lobsim_errors": (C.c_int, [vp, vp]),
        "lobsim_obs_dim": (C.c_int, [C.POINTER(abi.Cfg)]),
        "lobsim_action_dim": (C.c_int, [C.POINTER(abi.Cfg)]),
        "lobsim_launch_count": (i64, [vp]),
        "lobsim_kernel_path": (C.c_int, [vp]),
        "lobsim_source_hash": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    if L.lobsim_abi_version() != abi.ABI_VERSION:
        raise LobsimError("liblobsim.so ABI version mismatch: rebuild")
    from .build import source_hash

    built_from, here = L.lobsim_source_hash().decode(), source_hash()
    if built_from != here and native == _NATIVE:
        raise LobsimError(f"{_NATIVE} was built from other sources (stamp {built_from[:12]}, tree {here[:12]}): rebuild "
                          "(python -m rl4mm_b200.build, or __graft_entry__.build())")
    _LIB = L
    return L


EXPORTED_SYMBOLS = [
    "lobsim_last_error", "lobsim_abi_version", "lobsim_state_bytes", "lobsim_create", "lobsim_destroy",
    "lobsim_load_stream", "lobsim_reset", "lobsim_step", "lobsim_step_host", "lobsim_rollout", "lobsim_rollout_info", "lobsim_rollout_agents", "lobsim_replay",
    "lobsim_replay_host", "lobsim_forward_step", "lobsim_set_book", "lobsim_reset_book", "lobsim_process_orders", "lobsim_submit_orders_dev", "lobsim_dump_book",
    "lobsim_dump_agent_orders", "lobsim_get_depth_dev", "lobsim_get_agent_orders_dev", "lobsim_get_book_dev",
    "lobsim_set_book_dev", "lobsim_get_state", "lobsim_get_state_dev", "lobsim_get_fills", "lobsim_errors",
    "lobsim_obs_dim", "lobsim_action_dim", "lobsim_launch_count", "lobsim_kernel_path", "lobsim_source_hash",
]


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().lobsim_last_error().decode(errors="replace")
        raise LobsimError(f"lobsim call failed ({rc}): {msg}")


def np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
