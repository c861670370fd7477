"""ctypes / numpy mirror of ``include/lobsim.h`` (the C ABI of the device library).

Kept in one place so the host façade, the tests and the CPU oracle's wrapper all describe the same bytes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 1
MAX_FEATURES = 16

# return codes
OK, E_INVALID, E_CUDA, E_NOMEM, E_STATE = 0, -1, -2, -3, -4

# per-env sticky error bits
ERR_EMPTY_BOOK = 1
ERR_LEVEL_OVERFLOW = 2
ERR_ORDER_OVERFLOW = 4
ERR_AGENT_OVERFLOW = 8
ERR_BAD_VOLUME = 16
ERR_NO_SNAPSHOT = 32
ERR_END_OF_STREAM = 64
ERR_FILL_LOG_FULL = 128
ERR_AUM_NONPOSITIVE = 256
ERR_BAD_ACTION = 512
ERR_NAMES = {
    ERR_EMPTY_BOOK: "EMPTY_BOOK", ERR_LEVEL_OVERFLOW: "LEVEL_OVERFLOW", ERR_ORDER_OVERFLOW: "ORDER_OVERFLOW",
    ERR_AGENT_OVERFLOW: "AGENT_OVERFLOW", ERR_BAD_VOLUME: "BAD_VOLUME", ERR_NO_SNAPSHOT: "NO_SNAPSHOT",
    ERR_END_OF_STREAM: "END_OF_STREAM", ERR_FILL_LOG_FULL: "FILL_LOG_FULL", ERR_AUM_NONPOSITIVE: "AUM_NONPOSITIVE",
    ERR_BAD_ACTION: "BAD_ACTION",
}

MSG_LIMIT, MSG_CANCEL, MSG_DELETE, MSG_MARKET = 1, 2, 3, 4
BUY, SELL = 0, 1
REF_AGGREGATE = 0
REF_AGENT = 0x80000000
NO_PRICE = -(2**31)

FEAT_SPREAD, FEAT_BOOK_IMBALANCE, FEAT_PRICE_MOVE, FEAT_PRICE_RANGE, FEAT_VOLATILITY, FEAT_PRICE = range(6)
FEAT_TRADE_DIR_IMBALANCE, FEAT_TRADE_VOL_IMBALANCE, FEAT_INVENTORY, FEAT_EPISODE_PROPORTION, FEAT_TIME_OF_DAY = range(
    6, 11
)
REWARD_PNL, REWARD_INV_ADJ_PNL, REWARD_ROLLING_SHARPE = 0, 1, 2
MAX_SHARPE_WINDOW = 256
FEAT_AMIHUD_LAMBDA = 11
INFO_FIELDS = ("asset_price", "inventory", "cash", "aum", "market_spread", "best_buy", "best_sell", "err")
INFO_DIM = len(INFO_FIELDS)
AGENT_NONE, AGENT_FIXED, AGENT_TERADACTYL, AGENT_EXTERNAL, AGENT_RANDOM = 0, 1, 2, 3, 4
PATH_GENERAL, PATH_FAST, PATH_DEEP = 0, 1, 2
# per-env outcome of lobsim_set_book_dev / LobSim.set_books, in the order the checks run (the first that fails is reported)
SETBOOK_OK, SETBOOK_SKIPPED = 0, 1
SETBOOK_E_COUNT, SETBOOK_E_VOLUME, SETBOOK_E_UNSORTED, SETBOOK_E_LEVELS, SETBOOK_E_ORDERS, SETBOOK_E_AGENTS = range(-1, -7, -1)

MSG_DTYPE = np.dtype([("price", "<i4"), ("volume", "<i4"), ("ref", "<u4"), ("meta", "<u4")])
assert MSG_DTYPE.itemsize == 16


def meta(msg_type, direction):
    return np.uint32(msg_type) | (np.uint32(direction) << np.uint32(3))


class Feature(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("lookback", C.c_int32), ("update_us", C.c_int64), ("min_value", C.c_double),
        ("max_value", C.c_double), ("iparam", C.c_int32), ("norm_len", C.c_int32), ("dparam", C.c_double),
    ]


class Reward(C.Structure):
    _fields_ = [("kind", C.c_int32), ("asymmetric", C.c_int32), ("inventory_aversion", C.c_double)]


class Agent(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("inventory_index", C.c_int32), ("fixed_action", C.c_double * 5),
        ("max_inventory", C.c_double), ("default_kappa", C.c_double), ("default_omega", C.c_double),
        ("max_kappa", C.c_double), ("exponent", C.c_double), ("market_clearing", C.c_int32), ("reserved", C.c_int32),
    ]


class Cfg(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("n_envs", C.c_int32), ("n_levels", C.c_int32), ("tick_size", C.c_int32),
        ("step_us", C.c_int64), ("episode_steps", C.c_int32), ("warmup_steps", C.c_int32),
        ("min_quote_level", C.c_int32), ("max_quote_level", C.c_int32), ("outer_levels", C.c_int32),
        ("resync", C.c_int32), ("active_volume", C.c_int32), ("market_order_clearing", C.c_int32),
        ("enter_spread", C.c_int32), ("inc_prev_action_in_obs", C.c_int32), ("portfolio_carryover", C.c_int32),
        ("n_features", C.c_int32), ("concentration", C.c_double), ("market_order_fraction_of_inventory", C.c_double),
        ("initial_cash", C.c_double), ("initial_inventory", C.c_int64), ("features", Feature * MAX_FEATURES),
        ("step_reward", Reward), ("terminal_reward", Reward), ("max_levels_per_side", C.c_int32),
        ("max_orders_per_side", C.c_int32), ("max_agent_orders", C.c_int32), ("fill_log_capacity", C.c_int32),
    ]


class Stream(C.Structure):
    _fields_ = [
        ("msgs", C.c_void_p), ("n_msgs", C.c_uint64), ("step_off", C.c_void_p), ("n_grid_steps", C.c_uint32),
        ("snapshots", C.c_void_p), ("snap_valid", C.c_void_p), ("n_seconds", C.c_uint32), ("reserved", C.c_uint32),
        ("t0_us", C.c_int64),
    ]


class Order(C.Structure):
    _fields_ = [
        ("env", C.c_int32), ("type", C.c_int32), ("direction", C.c_int32), ("price", C.c_int32),
        ("volume", C.c_int32), ("is_external", C.c_int32), ("ref", C.c_uint32), ("reserved", C.c_uint32),
    ]


ORDER_DTYPE = np.dtype(
    [("env", "<i4"), ("type", "<i4"), ("direction", "<i4"), ("price", "<i4"), ("volume", "<i4"),
     ("is_external", "<i4"), ("ref", "<u4"), ("reserved", "<u4")]
)
FILL_DTYPE = np.dtype(
    [("list", "<i4"), ("direction", "<i4"), ("price", "<i4"), ("volume", "<i4"), ("is_market", "<i4"), ("ref", "<u4")]
)
BOOK_ENTRY_DTYPE = np.dtype([("price", "<i4"), ("volume", "<i4"), ("ref", "<u4"), ("level", "<i4")])
ENV_STATE_DTYPE = np.dtype(
    [("inventory", "<i8"), ("cash", "<f8"), ("price", "<f8"), ("now_step", "<i4"), ("episode_start_step", "<i4"),
     ("min_buy_price", "<i4"), ("max_sell_price", "<i4"), ("best_buy", "<i4"), ("best_sell", "<i4"),
     ("best_buy_volume", "<i4"), ("best_sell_volume", "<i4"), ("err", "<u4"), ("stream_id", "<i4"),
     ("n_agent_orders", "<u4", (2,)), ("next_agent_id", "<u4"), ("reserved", "<u4")]
)
assert ORDER_DTYPE.itemsize == 32 and FILL_DTYPE.itemsize == 24 and BOOK_ENTRY_DTYPE.itemsize == 16
assert ENV_STATE_DTYPE.itemsize == 80, ENV_STATE_DTYPE.itemsize


def _order_field(x, shape, device):
    """One field of pack_orders as int32 [N, K]: a tensor (broadcast) or a scalar; values are taken modulo 2^32 (refs >= 2^31)."""
    import torch

    if isinstance(x, torch.Tensor):
        if x.dtype.is_floating_point or x.dtype.is_complex:
            raise TypeError(f"pack_orders: integer tensors only, got {x.dtype}")
        v = x.to(torch.int64)
        v = torch.where(v >= 2**31, v - 2**32, v).to(torch.int32)
        return v.expand(shape)
    x = int(x)
    return torch.full(shape, x - 2**32 if x >= 2**31 else x, dtype=torch.int32, device=device)


def pack_orders(type, direction, price, volume, is_external=0, ref=0):
    """The orders of N envs, K per env, as the int32 tensor [N, K, 8] that is a ``lobsim_order_t`` array in ORDER_DTYPE field
    order (the input of ``LobSim.submit_orders``).  Each argument is an integer tensor of shape [N, K] (or broadcastable to it)
    or a scalar; the tensors must be on one device, which the result is on, and at least one must be given.  ``env`` is set to
    the row index, so that the rows concatenated env by env are also a valid ``process_orders`` list; ``reserved`` is 0."""
    import torch

    fields = (type, direction, price, volume, is_external, ref)
    tensors = [f for f in fields if isinstance(f, torch.Tensor)]
    if not tensors:
        raise ValueError("pack_orders: at least one argument must be an [N, K] tensor")
    device = tensors[0].device
    if any(t.device != device for t in tensors):
        raise ValueError("pack_orders: all tensors must be on one device")
    shape = torch.broadcast_shapes(*(t.shape for t in tensors))
    if len(shape) != 2:
        raise ValueError(f"pack_orders: the fields must broadcast to [N, K], got {tuple(shape)}")
    n, k = shape
    env = torch.arange(n, dtype=torch.int32, device=device)[:, None].expand(n, k)
    cols = [env] + [_order_field(f, shape, device) for f in fields] + [torch.zeros(shape, dtype=torch.int32, device=device)]
    return torch.stack(cols, dim=-1).contiguous()


def default_cfg(**kw) -> Cfg:
    """A Cfg with the reference's defaults (HOE.py:54-81, OrderbookSimulator.py:24-35); override with kwargs."""
    cfg = Cfg()
    cfg.abi_version = ABI_VERSION
    cfg.n_envs = 1
    cfg.n_levels = 50
    cfg.tick_size = 100
    cfg.step_us = 100_000
    cfg.episode_steps = 18_000
    cfg.warmup_steps = 0
    cfg.min_quote_level, cfg.max_quote_level = 0, 10
    cfg.outer_levels = 20
    cfg.resync = 1
    cfg.active_volume = 100
    cfg.portfolio_carryover = 1
    cfg.concentration = -1.0
    cfg.initial_cash = 1000.0
    cfg.initial_inventory = 0
    cfg.step_reward = Reward(REWARD_INV_ADJ_PNL, 0, 1e-4)
    cfg.terminal_reward = Reward(REWARD_INV_ADJ_PNL, 0, 0.1)
    cfg.max_levels_per_side = 128
    cfg.max_orders_per_side = 512
    cfg.max_agent_orders = 64
    cfg.fill_log_capacity = 0
    feats = kw.pop("features", None)
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    if feats is not None:
        set_features(cfg, feats)
    return cfg


def set_features(cfg: Cfg, feats) -> None:
    if len(feats) > MAX_FEATURES:
        raise ValueError(f"at most {MAX_FEATURES} features")
    cfg.n_features = len(feats)
    for i, f in enumerate(feats):
        cfg.features[i] = f


def feature(kind, lookback=0, update_us=100_000, min_value=0.0, max_value=0.0, iparam=0, dparam=0.0, norm_len=0) -> Feature:
    """norm_len > 0 switches on the rolling z-score (normalisation_on=True with max_norm_len=norm_len)."""
    return Feature(kind, lookback, update_us, float(min_value), float(max_value), iparam, int(norm_len), float(dparam))


def rolling_sharpe(max_window_size: int = 120, min_window_size: int = 60) -> Reward:
    assert 2 <= min_window_size <= max_window_size <= MAX_SHARPE_WINDOW
    return Reward(REWARD_ROLLING_SHARPE, max_window_size | (min_window_size << 16), 0.0)


def amihud(true_lookback: int = 10, slowing_factor: int = 10, update_us: int = 100_000, min_value=0.0, max_value=1.0) -> Feature:
    return feature(FEAT_AMIHUD_LAMBDA, (true_lookback + 1) * slowing_factor, update_us, min_value, max_value, iparam=slowing_factor)


def action_dim(cfg: Cfg) -> int:
    return (2 if cfg.concentration >= 0 else 4) + (1 if cfg.market_order_clearing else 0)


def obs_dim(cfg: Cfg) -> int:
    return cfg.n_features + (action_dim(cfg) if cfg.inc_prev_action_in_obs else 0)
