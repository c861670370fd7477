"""Shared helpers of the parity tests: golden loading, configuration building, canonical dumps."""
from __future__ import annotations

import gzip
import json
from pathlib import Path

import numpy as np

from rl4mm_b200 import abi
from rl4mm_b200.packing import PackedStream

GOLDEN = Path(__file__).resolve().parent / "golden"
REL_TOL = 1e-6  # north_star: features and rewards within 1e-6 relative
ABS_TOL = 1e-9


# hand-picked env configurations + seeded random ones, both produced by the unmodified reference (oracle/gen_golden.py)
ENV_GOLDEN_CASES = [("env_episodes.json.gz", i) for i in range(14)] + [("env_random.json.gz", i) for i in range(16)] + \
    [("rolling_sharpe_1e12.json.gz", i) for i in range(2)]       # RollingSharpe at the reference's default cash (1e12)


def load_golden(name: str):
    with gzip.open(GOLDEN / name, "rb") as f:
        return json.loads(f.read().decode())


def load_fixture_stream(tie_order: str = "reference") -> PackedStream:
    z = np.load(GOLDEN / "msft_fixture_packed.npz")
    s = PackedStream(np.ascontiguousarray(z[f"msgs_{tie_order}"]), z["step_off"], z["snapshots"], z["snap_valid"],
                     int(z["t0_us"]), int(z["step_us"]), 50, z["ext_ids"], "MSFT", "2012-06-21")
    s.validate()
    return s


_KINDS = {
    "SPREAD": abi.FEAT_SPREAD, "BOOK_IMBALANCE": abi.FEAT_BOOK_IMBALANCE, "PRICE_MOVE": abi.FEAT_PRICE_MOVE,
    "PRICE_RANGE": abi.FEAT_PRICE_RANGE, "VOLATILITY": abi.FEAT_VOLATILITY, "PRICE": abi.FEAT_PRICE,
    "TRADE_DIR_IMBALANCE": abi.FEAT_TRADE_DIR_IMBALANCE, "TRADE_VOL_IMBALANCE": abi.FEAT_TRADE_VOL_IMBALANCE,
    "INVENTORY": abi.FEAT_INVENTORY, "EPISODE_PROPORTION": abi.FEAT_EPISODE_PROPORTION,
    "TIME_OF_DAY": abi.FEAT_TIME_OF_DAY, "AMIHUD_LAMBDA": abi.FEAT_AMIHUD_LAMBDA,
}


def features_from_golden(specs):
    return [abi.feature(_KINDS[d["kind"]], d["lookback"], d["update_us"], d["min"], d["max"], d.get("iparam", 0),
                        d.get("dparam", 0.0), d.get("norm_len", 0)) for d in specs]


def reward_from_golden(spec) -> abi.Reward:
    if spec[0] == "PnL":
        return abi.Reward(abi.REWARD_PNL, 0, 0.0)
    if spec[0] == "RS":
        return abi.rolling_sharpe(spec[1], spec[2])
    return abi.Reward(abi.REWARD_INV_ADJ_PNL, int(spec[2]), float(spec[1]))


def cfg_from_env_case(case, n_envs: int = 1, **kw) -> abi.Cfg:
    ek = case["env_kwargs"]
    feats = features_from_golden(case["features"])
    return abi.default_cfg(
        n_envs=n_envs, n_levels=50, episode_steps=case["episode_steps"], warmup_steps=case["warmup_steps"],
        outer_levels=case["outer_levels"], min_quote_level=ek.get("min_quote_level", 0),
        max_quote_level=ek.get("max_quote_level", 10), market_order_clearing=int(ek.get("market_order_clearing", False)),
        market_order_fraction_of_inventory=float(ek.get("market_order_fraction_of_inventory", 0.0)),
        enter_spread=int(ek.get("enter_spread", False)),
        inc_prev_action_in_obs=int(ek.get("inc_prev_action_in_obs", False)),
        concentration=float(ek["concentration"]) if ek.get("concentration") is not None else -1.0,
        initial_inventory=int(case["portfolio"][0]), initial_cash=float(case["portfolio"][1]),
        step_reward=reward_from_golden(case["reward_step"]), terminal_reward=reward_from_golden(case["reward_term"]),
        features=feats, fill_log_capacity=256, **kw,
    )


CAPACITY_BITS = abi.ERR_LEVEL_OVERFLOW | abi.ERR_ORDER_OVERFLOW | abi.ERR_AGENT_OVERFLOW | abi.ERR_FILL_LOG_FULL


def exceeded_bits(peaks: dict, cfg: abi.Cfg) -> int:
    """The capacity error bits that an unbounded book with these high-water marks (oracle.Oracle.peaks) earns on a device book
    with the capacities of ``cfg``: more levels, orders or agent orders on a side than it holds, more fills in one call than the
    fill log holds."""
    bits = 0
    if max(peaks["levels"]) > cfg.max_levels_per_side:
        bits |= abi.ERR_LEVEL_OVERFLOW
    if max(peaks["orders"]) > cfg.max_orders_per_side:
        bits |= abi.ERR_ORDER_OVERFLOW
    if max(peaks["agents"]) > cfg.max_agent_orders:
        bits |= abi.ERR_AGENT_OVERFLOW
    if cfg.fill_log_capacity > 0 and peaks["fills"] > cfg.fill_log_capacity:
        bits |= abi.ERR_FILL_LOG_FULL
    return bits


def capacity_excluded(err, oracle, cfg: abi.Cfg, what="") -> bool:
    """True when the device flagged a capacity bit for this env, so that it leaves the comparison -- after checking that the flag
    is justified: the oracle (unbounded) went over at least one capacity since the error bits were last cleared.  A kernel that
    raised a capacity flag by mistake would otherwise drop the env from the test silently."""
    bits = int(err) & CAPACITY_BITS
    if not bits:
        return False
    peaks = oracle.peaks()
    assert exceeded_bits(peaks, cfg), (what, f"capacity bits {bits:#x} without a capacity exceeded", peaks)
    return True


def canon_book(entries: np.ndarray, ext_ids: np.ndarray | None = None):
    """lobsim_book_entry_t[] -> [[price, volume, kind, ext_id]] (kind 0 aggregate, 1 external, 2 agent)."""
    out = []
    for e in entries:
        ref = int(e["ref"])
        if ref & abi.REF_AGENT:
            out.append([int(e["price"]), int(e["volume"]), 2, 0])
        elif ref == abi.REF_AGGREGATE:
            out.append([int(e["price"]), int(e["volume"]), 0, 0])
        else:
            out.append([int(e["price"]), int(e["volume"]), 1, int(ext_ids[ref]) if ext_ids is not None else ref])
    return out


def canon_fills(fills: np.ndarray):
    """lobsim_fill_t[] (emission order) -> the reference's two lists, internal first then external."""
    rows = [[int(f["list"]), int(f["direction"]), int(f["price"]), int(f["volume"]), int(f["is_market"])] for f in fills]
    return [r for r in rows if r[0] == 0] + [r for r in rows if r[0] == 1]


def close(a, b, rel=REL_TOL, abs_=ABS_TOL) -> bool:
    a, b = float(a), float(b)
    if np.isnan(a) or np.isnan(b):
        return np.isnan(a) and np.isnan(b)
    return abs(a - b) <= abs_ + rel * max(abs(a), abs(b))


def reward_close(got, step) -> bool:
    """Reward of a golden env step.  1e-6 relative -- except for the RollingSharpe steps of rolling_sharpe_1e12.json.gz, which carry
    the first-order bound on |delta reward| between two implementations whose log() is good to one ulp (``bound``,
    oracle/gen_golden.py::golden_rolling_sharpe_1e12): at 1e12 cash the reference's own reward is only defined up to that."""
    if close(got, step["reward"]):
        return True
    b = step.get("bound")
    return b is not None and abs(float(got) - step["reward"]) <= b


def assert_close_vec(actual, expected, what=""):
    assert len(actual) == len(expected), what
    for i, (a, b) in enumerate(zip(actual, expected)):
        assert close(a, b), f"{what}[{i}]: {a!r} != {b!r}"


def snapshot_stream(levels, n_levels: int = 50, step_us: int = 100_000) -> PackedStream:
    """A message-free one-second stream whose snapshot at second 0 holds ``levels`` = [[side, price, volume], ...]."""
    snaps = np.zeros((2, 2, n_levels, 2), np.int32)
    snaps[..., 0] = abi.NO_PRICE
    for side in (0, 1):
        lv = sorted([l for l in levels if l[0] == side], key=lambda l: -l[1] if side == 0 else l[1])
        for i, (_, p, v) in enumerate(lv):
            snaps[:, side, i] = (p, v)
    n_grid = 1_000_000 // step_us
    s = PackedStream(np.zeros(0, abi.MSG_DTYPE), np.zeros(n_grid + 1, np.uint32), snaps, np.ones(2, np.uint8), 0,
                     step_us, n_levels)
    s.validate()
    return s


# ---- evaluation path (tests/golden/episode_summary.json.gz) -----------------------------------------------------------
def summary_case_cfg(case, n_envs: int = 1) -> abi.Cfg:
    """The env of oracle/gen_golden.py::golden_episode_summary: features [Spread, Inventory], PnL rewards, L=50."""
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 100 * 100), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -100000, 100000)]
    return abi.default_cfg(n_envs=n_envs, n_levels=50, episode_steps=case["episode_steps"], warmup_steps=0, features=feats,
                           step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
                           initial_cash=float(case["initial_cash"]), initial_inventory=0, portfolio_carryover=1)


def summary_case_agent(case) -> abi.Agent:
    import ctypes

    a = case["agent"]
    if a["kind"] == "fixed":
        return abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(*(list(map(float, a["action"])) + [0.0])))
    return abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=a["inventory_index"], max_inventory=float(a["max_inventory"]),
                     default_kappa=a["default_kappa"], default_omega=a["default_omega"], max_kappa=a["max_kappa"],
                     exponent=a["exponent"], market_clearing=0)


def assert_summary_matches(esd, case, sharpes):
    exp = case["esd"]
    assert set(esd) == set(exp)
    for key in exp:
        assert len(esd[key]) == len(exp[key]) == case["n_iterations"], key
        for e, (got, want) in enumerate(zip(esd[key], exp[key])):
            assert_close_vec(np.atleast_1d(np.asarray(got, dtype=float)), np.atleast_1d(np.asarray(want, dtype=float)), f"{case['name']} {key}[{e}]")
    assert_close_vec(np.asarray(sharpes, dtype=float), np.asarray(case["sharpe"], dtype=float), "sharpe")
