"""The batched order submission without a CUDA device: the C entry point is exported with its argument types and rejects null
and out-of-range arguments, the façade raises instead of falling back to a host path, and abi.pack_orders builds exactly the
bytes of a lobsim_order_t array."""
import ctypes as C

import numpy as np
import pytest

from rl4mm_b200 import abi


@pytest.fixture(scope="module")
def lobsim_lib():
    from rl4mm_b200.build import build_all

    build_all()
    from rl4mm_b200._lib import lib

    return lib()


def test_submit_entry_point_validates_without_a_device(lobsim_lib):
    from rl4mm_b200._lib import EXPORTED_SYMBOLS

    assert "lobsim_submit_orders_dev" in EXPORTED_SYMBOLS
    fn = lobsim_lib.lobsim_submit_orders_dev
    assert fn.restype is C.c_int
    assert fn.argtypes == [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                           C.c_void_p]
    buf = (C.c_int64 * 64)()
    ptr = C.cast(buf, C.c_void_p)
    assert fn(None, 4, ptr, ptr, ptr, 0, None, ptr, None) == abi.E_INVALID
    assert b"null" in lobsim_lib.lobsim_last_error()


def test_submit_facade_has_no_cpu_fallback(lobsim_lib):
    import torch

    from rl4mm_b200._lib import LobsimError

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from rl4mm_b200.device import LobSim

    with pytest.raises(LobsimError):
        LobSim(abi.default_cfg(n_envs=2)).submit_orders(torch.zeros((2, 4, 8), dtype=torch.int32))


def test_pack_orders_is_a_lobsim_order_array():
    import torch

    rng = np.random.default_rng(3)
    N, K = 5, 7
    typ = rng.integers(0, 6, size=(N, K))
    side = rng.integers(0, 2, size=(N, K))
    price = rng.integers(-(2**31), 2**31, size=(N, K))
    vol = rng.integers(-5, 1000, size=(N, K))
    ext = rng.integers(0, 2, size=(N, K))
    ref = rng.integers(0, 2**32, size=(N, K), dtype=np.uint64)
    ref[0, 0] = 0xFFFFFFFF
    want = np.zeros((N, K), abi.ORDER_DTYPE)
    want["env"] = np.arange(N)[:, None]
    want["type"], want["direction"], want["price"], want["volume"], want["is_external"], want["ref"] = typ, side, price, vol, ext, ref
    got = abi.pack_orders(*(torch.tensor(x.astype(np.int64)) for x in (typ, side, price, vol, ext, ref)))
    assert got.dtype == torch.int32 and tuple(got.shape) == (N, K, 8) and got.is_contiguous()
    assert got.numpy().tobytes() == want.tobytes()
    # scalars broadcast against the tensors; any integer dtype
    got = abi.pack_orders(abi.MSG_LIMIT, torch.tensor(side, dtype=torch.int8), torch.tensor(price), 17, ref=0xFFFFFFFF)
    w2 = np.zeros((N, K), abi.ORDER_DTYPE)
    w2["env"] = np.arange(N)[:, None]
    w2["type"], w2["direction"], w2["price"], w2["volume"], w2["ref"] = abi.MSG_LIMIT, side, price, 17, 0xFFFFFFFF
    assert got.numpy().tobytes() == w2.tobytes()
    # a [1, K] row broadcast against [N, 1]
    got = abi.pack_orders(torch.full((1, K), abi.MSG_MARKET), torch.zeros((N, 1), dtype=torch.int32), 0, torch.ones((N, K), dtype=torch.int64))
    assert tuple(got.shape) == (N, K, 8) and np.all(got.numpy()[..., 1] == abi.MSG_MARKET)
    with pytest.raises(ValueError):
        abi.pack_orders(1, 0, 100, 5)                                            # no tensor: N and K unknown
    with pytest.raises(ValueError):
        abi.pack_orders(torch.ones(3, dtype=torch.int32), 0, 100, 5)             # not [N, K]
    with pytest.raises(TypeError):
        abi.pack_orders(torch.ones((2, 2)), 0, 100, 5)                           # float tensor
