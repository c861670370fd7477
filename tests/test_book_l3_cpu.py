"""The batched L3 read and write without a CUDA device: both C entry points are exported and reject null arguments, and the
façade raises instead of falling back to a host path."""
import ctypes as C

import pytest

from rl4mm_b200 import abi


@pytest.fixture(scope="module")
def lobsim_lib():
    from rl4mm_b200.build import build_all

    build_all()
    from rl4mm_b200._lib import lib

    return lib()


def test_entry_points_are_exported():
    from rl4mm_b200._lib import EXPORTED_SYMBOLS

    assert "lobsim_get_book_dev" in EXPORTED_SYMBOLS and "lobsim_set_book_dev" in EXPORTED_SYMBOLS


def test_entry_points_validate_without_a_device(lobsim_lib):
    buf = (C.c_int64 * 16)()
    ptr = C.cast(buf, C.c_void_p)
    assert lobsim_lib.lobsim_get_book_dev(None, 1, ptr, ptr, None) == abi.E_INVALID
    assert b"null" in lobsim_lib.lobsim_last_error()
    assert lobsim_lib.lobsim_set_book_dev(None, 1, ptr, ptr, ptr, None) == abi.E_INVALID
    assert b"null" in lobsim_lib.lobsim_last_error()


def test_status_codes_in_check_order():
    assert (abi.SETBOOK_OK, abi.SETBOOK_SKIPPED) == (0, 1)
    assert [abi.SETBOOK_E_COUNT, abi.SETBOOK_E_VOLUME, abi.SETBOOK_E_UNSORTED, abi.SETBOOK_E_LEVELS, abi.SETBOOK_E_ORDERS,
            abi.SETBOOK_E_AGENTS] == [-1, -2, -3, -4, -5, -6]


def test_book_l3_facade_has_no_cpu_fallback(lobsim_lib):
    import torch

    from rl4mm_b200._lib import LobsimError
    from rl4mm_b200.device import LobSim

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(LobsimError):
        LobSim(abi.default_cfg(n_envs=2)).book_l3()
    with pytest.raises(LobsimError):
        LobSim(abi.default_cfg(n_envs=2)).set_books(torch.zeros((2, 2, 1, 4), dtype=torch.int32))
