"""The batched agent-order read without a CUDA device: the C entry point is exported with its argument types and rejects
its arguments, and the façade raises instead of falling back to a host path."""
import ctypes as C

import pytest

from rl4mm_b200 import abi


@pytest.fixture(scope="module")
def lobsim_lib():
    from rl4mm_b200.build import build_all

    build_all()
    from rl4mm_b200._lib import lib

    return lib()


def test_agent_orders_entry_point_validates_without_a_device(lobsim_lib):
    from rl4mm_b200._lib import EXPORTED_SYMBOLS

    assert "lobsim_get_agent_orders_dev" in EXPORTED_SYMBOLS
    fn = lobsim_lib.lobsim_get_agent_orders_dev
    assert fn.restype is C.c_int
    assert fn.argtypes == [C.c_void_p, C.c_int32] + [C.c_void_p] * 8
    buf = (C.c_int64 * 8)()
    ptr = C.cast(buf, C.c_void_p)
    assert fn(None, 1, ptr, ptr, ptr, ptr, None, None, None, None) == abi.E_INVALID
    assert b"null" in lobsim_lib.lobsim_last_error()


def test_agent_orders_facade_has_no_cpu_fallback(lobsim_lib):
    import torch

    from rl4mm_b200._lib import LobsimError
    from rl4mm_b200.device import LobSim

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(LobsimError):
        LobSim(abi.default_cfg(n_envs=2)).agent_orders()
