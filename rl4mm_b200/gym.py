"""Mirror of ``rl4mm/gym``: ``HistoricalOrderbookEnvironment`` (batched), ``BetaOrderDistributor``,
``SimpleInfoCalculator`` and ``generate_trajectory``.

The env keeps the reference's constructor arguments (rl4mm/gym/HistoricalOrderbookEnvironment.py:54-81) and the gym
0.21 API -- ``reset() -> obs``, ``step(action) -> (obs, reward, done, info)`` -- for ``n_envs`` books at once.  With
``n_envs == 1`` the return values have the reference's shapes (obs ``[F]``, float reward, bool done).  ``reset`` /
``step`` are one kernel launch each (csrc/lobsim.cu ``k_advance<true>``): action -> Beta ladders -> agent orders ->
history of the step -> fills / portfolio -> features -> reward, all on the device.
"""
from __future__ import annotations

import abc
from datetime import datetime, timedelta
from typing import List, Optional

import numpy as np

from . import abi
from .features import (EpisodeProportion, Feature, Inventory, Portfolio, PriceMove, Spread, TimeOfDay,
                       TradeDirectionImbalance, TradeVolumeImbalance, Volatility)
from .rewards import InventoryAdjustedPnL, RewardFunction
from .simulation import DeviceDatabase

EPS = 0.000001
TICK_SIZE = 100


class Box:
    """The part of ``gym.spaces.Box`` the reference uses (gym itself is not a dependency of this path)."""

    def __init__(self, low, high, shape=None, dtype=np.float64):
        if shape is not None:
            low, high = np.full(shape, low, dtype=dtype), np.full(shape, high, dtype=dtype)
        self.low, self.high = np.asarray(low, dtype=dtype), np.asarray(high, dtype=dtype)
        self.shape, self.dtype = self.low.shape, dtype
        self._rng = np.random.default_rng()

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)

    def sample(self):
        return self._rng.uniform(self.low, self.high)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


# ---- rl4mm/gym/action_interpretation/OrderDistributors.py ------------------------------------------------------------
class OrderDistributor(metaclass=abc.ABCMeta):
    def __init__(self, quote_levels: int = 10, active_volume: int = 100):
        self.quote_levels, self.active_volume = quote_levels, active_volume
        self.tick_range = range(0, quote_levels)

    def convert_action(self, action: np.ndarray):
        return self._convert_action(np.array(action, dtype=float) + EPS)

    @abc.abstractmethod
    def _convert_action(self, action: np.ndarray):
        pass


class BetaOrderDistributor(OrderDistributor):
    """Host-side twin of csrc/env.cuh ``beta_ladder_lane`` (used by the info calculator and for inspection): weights
    x^(a-1) (1-x)^(b-1) at the level midpoints, normalised (1/B(a,b) cancels), ``np.round`` half-to-even."""

    def __init__(self, quote_levels: int = 10, active_volume: int = 100, concentration: float = None):
        super().__init__(quote_levels, active_volume)
        self.c = concentration
        self.midpoints = 1 / self.quote_levels * np.array([i + 0.5 for i in range(self.quote_levels)])

    def _ladder(self, a, b):
        a, b = np.asarray(a, dtype=float)[..., None], np.asarray(b, dtype=float)[..., None]
        x = self.midpoints
        with np.errstate(all="ignore"):
            logw = np.where(a - 1 == 0, 0.0, (a - 1) * np.log(x)) + np.where(b - 1 == 0, 0.0, (b - 1) * np.log1p(-x))
        w = np.exp(logw - logw.max(axis=-1, keepdims=True))
        w = w / w.sum(axis=-1, keepdims=True)
        return np.round(w * self.active_volume).astype(int)

    def _convert_action(self, action: np.ndarray):
        n = action.shape[-1]
        assert (self.c is None and n in (4, 5)) or (self.c is not None and n in (2, 3)), \
            f"Concentration is set to {self.c} and the action taken is of length {n}"
        if self.c is not None:
            a_buy, b_buy, a_sell, b_sell = action[..., 0], self.c - action[..., 0] + EPS, action[..., 1], self.c - action[..., 1] + EPS
        else:
            a_buy, b_buy, a_sell, b_sell = action[..., 0], action[..., 1], action[..., 2], action[..., 3]
        return {"buy": self._ladder(a_buy, b_buy), "sell": self._ladder(a_sell, b_sell)}


# ---- rl4mm/gym/order_tracking/InfoCalculators.py ---------------------------------------------------------------------
class InfoCalculator(metaclass=abc.ABCMeta):
    @abc.abstractmethod
    def calculate(self, internal_state, action: np.ndarray):
        pass


class SimpleInfoCalculator(InfoCalculator):
    """InfoCalculators.py:21-89, vectorised over envs: ``internal_state`` is the structured array returned by
    ``LobSim.state()`` (price, inventory, cash, best prices); every value of the returned dict is an array [N]."""

    def __init__(self, market_order_fraction_of_inventory: float = 0.0, enter_spread: bool = False,
                 order_distributor: OrderDistributor = None, concentration: float = None):
        self.market_order_count = 0
        self.market_order_total_volume = 0
        self.market_order_fraction_of_inventory = market_order_fraction_of_inventory
        self.enter_spread = enter_spread
        self.order_distributor = order_distributor or BetaOrderDistributor(concentration=concentration)

    def calculate(self, internal_state, action: np.ndarray):
        st = internal_state
        action = np.atleast_2d(np.asarray(action, dtype=float))
        spread = (st["best_sell"].astype(np.int64) - st["best_buy"].astype(np.int64)).astype(float)
        orders = self.order_distributor.convert_action(action)
        total, n_levels = self.order_distributor.active_volume, self.order_distributor.quote_levels
        dist = np.arange(n_levels)
        best_buy, best_sell = np.sign(orders["buy"]).argmax(axis=-1), np.sign(orders["sell"]).argmax(axis=-1)
        midprice_offset = (best_sell - best_buy) / 2
        agent_spread = (best_buy + best_sell).astype(float)
        buy_com, sell_com = orders["buy"] @ dist / total, orders["sell"] @ dist / total
        weighted_offset, weighted_spread = (sell_com - buy_com) / 2, buy_com + sell_com
        if not self.enter_spread:
            agent_spread = agent_spread + spread
            weighted_spread = weighted_spread + spread
        inv = st["inventory"].astype(np.int64)
        info = dict(asset_price=st["price"].copy(), inventory=inv, cash=st["cash"].copy(),
                    aum=st["cash"] + st["price"] * inv, market_spread=spread, agent_spread=agent_spread,
                    agent_weighted_spread=weighted_spread, midprice_offset=midprice_offset,
                    weighted_midprice_offset=weighted_offset)
        n = action.shape[-1]
        if n in (2, 3):
            info["bid_action"], info["ask_action"] = action[:, [0]], action[:, [1]]
        elif n in (4, 5):
            info["bid_action"], info["ask_action"] = action[:, [0, 1]], action[:, [2, 3]]
        else:
            raise NotImplementedError("Action dim should be 2, 3, 4, 5 based on current options.")
        if n in (3, 5):
            info["market_order_action"] = action[:, [-1]]
            hit = np.abs(inv) > action[:, -1]
            self.market_order_count = self.market_order_count + hit.astype(int)
            self.market_order_total_volume = self.market_order_total_volume + np.where(
                hit, np.round(np.abs(inv) * self.market_order_fraction_of_inventory), 0)
        info["market_order_count"] = self.market_order_count
        info["market_order_total_volume"] = self.market_order_total_volume
        return info


# ---- rl4mm/gym/HistoricalOrderbookEnvironment.py -----------------------------------------------------------------------
class HistoricalOrderbookEnvironment:
    metadata = {"render.modes": ["human"]}

    def __init__(
        self,
        features: List[Feature] = None,
        max_distribution_param: float = 10.0,
        ticker: str = "MSFT",
        step_size: timedelta = timedelta(seconds=0.1),
        episode_length: timedelta = timedelta(minutes=30),
        initial_portfolio: Portfolio = None,
        min_quote_level: int = 0,
        max_quote_level: int = 10,
        min_date: datetime = datetime(2019, 1, 2),
        max_date: datetime = datetime(2019, 1, 2),
        min_start_timedelta: timedelta = timedelta(hours=10),
        max_end_timedelta: timedelta = timedelta(hours=15, minutes=30),
        simulator=None,
        market_order_clearing: bool = False,
        inc_prev_action_in_obs: bool = False,
        max_inventory: int = 100000,
        per_step_reward_function: RewardFunction = None,
        terminal_reward_function: RewardFunction = None,
        info_calculator: InfoCalculator = None,
        order_distributor: OrderDistributor = None,
        concentration: Optional[float] = None,
        market_order_fraction_of_inventory: float = 0.0,
        enter_spread: bool = False,
        n_levels: int = 50,
        preload_orders: bool = True,
        *,
        n_envs: int = 1,
        database: DeviceDatabase = None,
        outer_levels: int = 20,
        device: int = 0,
        seed: Optional[int] = None,
        start_rng: str = "generator",
        auto_reset: bool = False,
        on_error: str = "raise",
        portfolio_carryover: bool = True,
        max_levels_per_side: int = 128,
        max_orders_per_side: int = 512,
        max_agent_orders: int = 64,
        fill_log_capacity: int = 0,
    ):
        if simulator is not None and database is None:
            database = simulator.database
            n_levels, outer_levels = simulator.n_levels, simulator.outer_levels
        assert database is not None and len(database.streams) > 0, "a DeviceDatabase with packed stream(s) is required"
        if concentration is not None:
            assert order_distributor is None, "When specifying concentration, no order distributor should be passed."
            assert concentration >= max_distribution_param, "Concentration is less than max_distribution_param."
            self.action_space = Box(low=0.0, high=concentration, shape=(2,), dtype=np.float64)
        else:
            self.action_space = Box(low=0.0, high=max_distribution_param, shape=(4,), dtype=np.float64)
        if market_order_clearing:
            self.action_space = Box(low=np.append(self.action_space.low, [0.0]),
                                    high=np.append(self.action_space.high, [max_inventory]), dtype=np.float64)
        self.max_distribution_param, self.ticker, self.step_size = max_distribution_param, ticker, step_size
        self.min_quote_level, self.max_quote_level = min_quote_level, max_quote_level
        assert episode_length % step_size == timedelta(0), "Episode length must be a multiple of step size!"
        self.n_steps = int(episode_length / step_size)
        self.episode_length = episode_length
        self.initial_portfolio = initial_portfolio or Portfolio(inventory=0, cash=1000)
        self.min_date, self.max_date = min_date, max_date
        self.min_start_timedelta, self.max_end_timedelta = min_start_timedelta, max_end_timedelta
        self.order_distributor = order_distributor or BetaOrderDistributor(max_quote_level - min_quote_level,
                                                                           concentration=concentration)
        self.market_order_clearing = market_order_clearing
        self.market_order_fraction_of_inventory = market_order_fraction_of_inventory
        self.per_step_reward_function = per_step_reward_function or InventoryAdjustedPnL(inventory_aversion=10 ** (-4))
        self.terminal_reward_function = terminal_reward_function or InventoryAdjustedPnL(inventory_aversion=0.1)
        self.enter_spread, self.n_levels, self.info_calculator = enter_spread, n_levels, info_calculator
        self._check_params()
        self.max_inventory = max_inventory
        self.features = features or self.get_default_features(step_size, episode_length)
        self.inc_prev_action_in_obs = inc_prev_action_in_obs
        low_obs = np.array([np.float32(f.min_value) for f in self.features])
        high_obs = np.array([np.float32(f.max_value) for f in self.features])
        if inc_prev_action_in_obs:
            low_obs = np.concatenate((low_obs, np.float32(self.action_space.low)))
            high_obs = np.concatenate((high_obs, np.float32(self.action_space.high)))
        self.observation_space = Box(low=low_obs, high=high_obs, dtype=np.float32)
        self.max_feature_window_size = max([f.window_size for f in self.features])
        self.n_envs, self.database = n_envs, database
        self.np_random = np.random.default_rng(seed)
        # "generator": episode starts from this env's own seeded Generator (vectorised for a batch); "numpy_global": drawn from
        # numpy's GLOBAL state with the reference's own call sequence (HOE.py:196,333-351), so that a run seeded with
        # np.random.seed(k) starts its episodes exactly where the reference would (one draw pair per env, env 0 first)
        assert start_rng in ("generator", "numpy_global")
        self.start_rng = start_rng
        # batched envs (n_envs > 1), vector-env conventions on top of the reference's single-env API: auto_reset -- an env whose episode
        # ended (done) or died (EmptyOrderbookError, overflow, ...) is reset inside step(): its returned observation is the first one of
        # the new episode, the last one of the old episode goes to info["terminal_observation"]; on_error="flag" -- device errors
        # do not raise for the whole batch but are reported per env in info["err"] (lobsim error bits)
        assert on_error in ("raise", "flag")
        self.auto_reset, self.on_error = auto_reset, on_error
        self._squeeze = n_envs == 1

        from .device import LobSim

        cfg = abi.default_cfg(
            n_envs=n_envs, n_levels=n_levels, tick_size=TICK_SIZE, step_us=step_size // timedelta(microseconds=1),
            episode_steps=self.n_steps, warmup_steps=int(self.max_feature_window_size / step_size),
            min_quote_level=min_quote_level, max_quote_level=max_quote_level, outer_levels=outer_levels,
            active_volume=self.order_distributor.active_volume, market_order_clearing=int(market_order_clearing),
            enter_spread=int(enter_spread), inc_prev_action_in_obs=int(inc_prev_action_in_obs),
            portfolio_carryover=int(portfolio_carryover),
            concentration=-1.0 if concentration is None else float(concentration),
            market_order_fraction_of_inventory=float(market_order_fraction_of_inventory or 0.0),
            initial_cash=float(self.initial_portfolio.cash), initial_inventory=int(self.initial_portfolio.inventory),
            features=[f.to_abi() for f in self.features], step_reward=self.per_step_reward_function.to_abi(),
            terminal_reward=self.terminal_reward_function.to_abi(), max_levels_per_side=max_levels_per_side,
            max_orders_per_side=max_orders_per_side, max_agent_orders=max_agent_orders,
            fill_log_capacity=fill_log_capacity,
        )
        self.sim = LobSim(cfg, device)
        for i, s in enumerate(database.streams):
            self.sim.load_stream(i, s)
        self.episode_start_steps = np.zeros(n_envs, np.int32)
        self.stream_ids = np.zeros(n_envs, np.int32)

    # ---- gym API -----------------------------------------------------------------------------------------------------
    def reset(self, env_ids=None):
        n = self.n_envs if env_ids is None else len(env_ids)
        sids, starts = np.zeros(n, np.int32), np.zeros(n, np.int32)
        if n > 64 and self.min_date == self.max_date and self.start_rng == "generator":   # one trading day: draw all the offsets at once
            day = self._get_random_trading_day()
            sid = self.database.stream_id(self.ticker, day)
            step_us = self.step_size // timedelta(microseconds=1)
            max_offset_steps = int((self.max_end_timedelta - self.episode_length - self.min_start_timedelta) / self.step_size)
            off = self.np_random.integers(0, max_offset_steps, size=n) if max_offset_steps > 0 else np.zeros(n, np.int64)
            us = self.min_start_timedelta // timedelta(microseconds=1) + off.astype(np.int64) * step_us
            us -= us % 1_000_000                                  # start episode on the second, HOE.py:342
            sids[:] = sid
            starts[:] = self.database.step_of(sid, day) + us // step_us
        else:
            for i in range(n):
                start = self._get_random_start_time()
                sids[i] = self.database.stream_id(self.ticker, start)
                starts[i] = self.database.step_of(sids[i], start)
        idx = slice(None) if env_ids is None else np.asarray(env_ids)
        self.stream_ids[idx], self.episode_start_steps[idx] = sids, starts
        obs = self.sim.reset(sids, starts, env_ids=env_ids).cpu().numpy()
        self._raise_on_errors()
        return obs[0] if self._squeeze and env_ids is None else obs

    def step(self, action):
        import torch

        a = np.asarray(action, dtype=np.float64)
        a = a.reshape(self.n_envs, -1)
        obs, rew, done = self.sim.step(torch.from_numpy(a))
        obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        err = None
        if self.on_error == "raise":
            self._raise_on_errors()
        else:
            err = self.sim.errors()
        info = {}
        if self.info_calculator is not None:
            info = self.info_calculator.calculate(internal_state=self.sim.state(), action=a)
        if err is not None:
            info["err"] = err
        if self.auto_reset:
            dead = np.zeros(self.n_envs, bool) if err is None else (err & (abi.ERR_EMPTY_BOOK | abi.ERR_BAD_ACTION | abi.ERR_END_OF_STREAM | abi.ERR_NO_SNAPSHOT)) != 0
            ids = np.flatnonzero(done | dead)
            if len(ids):
                info["terminal_observation"] = {int(i): obs[i].copy() for i in ids}
                done = done | dead
                obs = obs.copy()
                obs[ids] = np.asarray(self.reset(env_ids=ids)).reshape(len(ids), -1)
        if self._squeeze:
            return obs[0], float(rew[0]), bool(done[0]), self._squeeze_info(info)
        return obs, rew, done, info

    @staticmethod
    def _squeeze_info(info: dict) -> dict:
        """n_envs == 1: the reference's info shapes (InfoCalculators.py:31-59) -- scalars for the per-env values and
        1-tuples of 1-D arrays for the action slices -- so that ``extract_array_from_infos`` / ``get_sharpe`` see a
        [T] series, not [T, 1].  Deviation kept on purpose: ``agent_weighted_spread`` is the computed value; the reference
        returns the literal ``[1]`` there (InfoCalculators.py:40)."""
        out = {}
        for k, v in info.items():
            a = np.asarray(v)
            if k in ("bid_action", "ask_action", "market_order_action"):
                out[k] = (a.reshape(-1),)
            elif a.ndim >= 1 and a.size == 1:
                out[k] = a.reshape(-1)[0].item()
            else:
                out[k] = v
        return out

    def step_torch(self, actions):
        """Hot-loop variant: torch CUDA tensors in and out, no host round trip, no error polling."""
        return self.sim.step(actions)

    def book_depth(self, depth: int, orders: bool = False, agent: bool = False, out=None, stream=None):
        """Depth observations: the L2 book of every env read on the device in one launch (``LobSim.book_depth``), torch
        CUDA tensors price int32 / volume int64 [n_envs, 2, depth] (+ orders, agent_volume when asked for).  Batched and
        not squeezed, also when n_envs == 1; no host round trip, so it may sit next to ``step_torch`` in a CUDA graph."""
        return self.sim.book_depth(depth, orders=orders, agent=agent, out=out, stream=stream)

    def agent_orders(self, max_orders=None, queue: bool = True, out=None, stream=None):
        """The agent's resting orders of every env and their queue positions, read on the device in one launch
        (``LobSim.agent_orders``): torch CUDA tensors count [n_envs, 2], price / volume / id [n_envs, 2, max_orders] (+ level,
        ahead_orders, ahead_volume with ``queue``).  Batched and not squeezed, also when n_envs == 1; no host round trip, so
        it may sit next to ``step_torch`` in a CUDA graph."""
        return self.sim.agent_orders(max_orders=max_orders, queue=queue, out=out, stream=stream)

    def rollout(self, agent, T: int):
        """``generate_trajectory`` (rl4mm/gym/utils.py:100-117) for T steps of every env, fused on the device when the
        agent has a device implementation (FixedActionAgent, Teradactyl); returns torch tensors obs, act, rew, done."""
        desc = agent.to_abi()
        if desc is None:
            raise NotImplementedError("agent has no device implementation: drive the env with step() / step_torch()")
        return self.sim.rollout(T, desc)

    def _raise_on_errors(self):
        err = self.sim.errors()
        if np.any(err & abi.ERR_EMPTY_BOOK):
            from .orderbook import EmptyOrderbookError

            raise EmptyOrderbookError(f"empty book side in env(s) {np.flatnonzero(err & abi.ERR_EMPTY_BOOK)[:8]}")
        if np.any(err & abi.ERR_NO_SNAPSHOT):
            raise AssertionError("There is no data before the episode start time")
        if np.any(err & abi.ERR_BAD_ACTION):
            raise ValueError(f"non-finite action / Beta ladder in env(s) {np.flatnonzero(err & abi.ERR_BAD_ACTION)[:8]}")
        bad = err & (abi.ERR_LEVEL_OVERFLOW | abi.ERR_ORDER_OVERFLOW | abi.ERR_AGENT_OVERFLOW | abi.ERR_END_OF_STREAM)
        if np.any(bad):
            names = sorted({n for b, n in abi.ERR_NAMES.items() for e in np.unique(bad) if e & b})
            raise RuntimeError("device book error flags: " + ", ".join(names))

    # ---- random episode start, HOE.py:196,333-351 ----------------------------------------------------------------------
    def _get_random_start_time(self):
        if self.start_rng == "numpy_global":
            days = sorted(d for d, t in zip(self.database.dates, self.database.tickers) if t == self.ticker)
            return reference_random_start_time(self.min_date, self.max_date, self.min_start_timedelta, self.max_end_timedelta,
                                               self.episode_length, self.step_size, days)
        return self._get_random_trading_day() + self._random_offset_timestamp()

    def _random_offset_timestamp(self):
        max_offset_steps = int((self.max_end_timedelta - self.episode_length - self.min_start_timedelta) / self.step_size)
        random_offset_steps = int(self.np_random.integers(0, max_offset_steps)) if max_offset_steps > 0 else 0
        ts = self.min_start_timedelta + random_offset_steps * self.step_size
        ts -= timedelta(microseconds=ts.microseconds)  # start episode on the second
        return ts

    def _get_random_trading_day(self):
        days = [d for d, t in zip(self.database.dates, self.database.tickers)
                if t == self.ticker and self.min_date.date() <= d.date() <= self.max_date.date()]
        assert days, f"no packed data for {self.ticker} between {self.min_date.date()} and {self.max_date.date()}"
        return days[int(self.np_random.integers(0, len(days)))]

    def seed(self, seed=42):
        self.np_random = np.random.default_rng(seed)
        return [seed]

    def render(self, mode="human"):
        pass

    # ---- views for inspection (env 0 unless stated) ----------------------------------------------------------------------
    def _exchange_view(self, env: int = 0):
        from .orderbook import Exchange

        ex = Exchange(self.ticker, sim=self.sim, env=env)
        ex.use_stream_ids(self.database.streams[int(self.stream_ids[env])].ext_ids)
        return ex

    @property
    def central_orderbook(self):
        return self._exchange_view().central_orderbook

    @property
    def internal_orderbook(self):
        return self._exchange_view().internal_orderbook

    def mark_to_market_value(self):
        st = self.sim.state()
        v = st["inventory"] * st["price"] + st["cash"]
        return float(v[0]) if self._squeeze else v

    def _check_params(self):
        assert self.min_start_timedelta + self.episode_length <= self.max_end_timedelta, "Episode is too long"
        assert self.max_quote_level - self.min_quote_level == self.order_distributor.quote_levels
        if (self.market_order_clearing and self.market_order_fraction_of_inventory <= 0.0) or (
            not self.market_order_clearing and (self.market_order_fraction_of_inventory is not None
                                                and self.market_order_fraction_of_inventory > 0.0)):
            raise Exception(f"market_order_fraction_of_inventory {self.market_order_fraction_of_inventory} must be "
                            "positive if and only if market order clearing is on")

    @staticmethod
    def get_default_features(step_size: timedelta, episode_length: timedelta, normalisation_on: bool = False):
        """HOE.py:396-440"""
        assert step_size <= timedelta(seconds=0.1), "Default features require a minimum step size of 0.1 seconds."
        n = normalisation_on
        return [
            Spread(update_frequency=step_size, normalisation_on=n),
            PriceMove(name="price_move_0.1_s", update_frequency=timedelta(seconds=0.1), lookback_periods=1, normalisation_on=n),
            PriceMove(name="price_move_10_s", update_frequency=timedelta(seconds=1), lookback_periods=10, normalisation_on=n),
            Volatility(name="volatility_1_min", update_frequency=timedelta(seconds=0.1), lookback_periods=int(10 * 60), normalisation_on=n),
            Volatility(name="volatility_5_min", update_frequency=timedelta(seconds=1), lookback_periods=int(5 * 60), normalisation_on=n),
            Inventory(update_frequency=step_size, normalisation_on=n),
            EpisodeProportion(update_frequency=step_size, episode_length=episode_length, normalisation_on=n),
            TimeOfDay(n_buckets=10, normalisation_on=n),
            TradeDirectionImbalance(update_frequency=timedelta(seconds=0.1), lookback_periods=int(60 * 10), normalisation_on=n),
            TradeVolumeImbalance(update_frequency=timedelta(seconds=0.1), lookback_periods=int(60 * 10), normalisation_on=n),
        ]


def reference_random_start_time(min_date, max_date, min_start_timedelta, max_end_timedelta, episode_length, step_size, trading_days):
    """``HistoricalOrderbookEnvironment._get_random_start_time`` (HOE.py:196,333-351) with the reference's own draws from numpy's
    GLOBAL random state, in the reference's order: ``np.random.choice(pd.bdate_range(min_date, max_date))`` (one bounded integer
    draw over the business days), mapped to the next trading day (here: the next day that has packed data, the role of
    ``get_next_trading_dt``), then ``np.random.randint(0, max_offset_steps)`` (no draw when the range is empty, :337-340);
    the start is floored to the whole second (:342)."""
    import pandas as pd

    bdays = pd.bdate_range(min_date, max_date)
    day = pd.Timestamp(np.random.choice(bdays)).to_pydatetime()
    day = datetime.combine(day.date(), datetime.min.time())
    later = [d for d in trading_days if d >= day]
    assert later, f"no packed data on or after {day.date()}"
    day = later[0]
    max_offset_steps = int((max_end_timedelta - episode_length - min_start_timedelta) / step_size)
    try:
        random_offset_steps = int(np.random.randint(low=0, high=max_offset_steps))
    except ValueError:
        random_offset_steps = 0
    ts = min_start_timedelta + random_offset_steps * step_size
    ts -= timedelta(microseconds=ts.microseconds)
    return day + ts


def generate_trajectory(agent, env):
    """rl4mm/gym/utils.py:100-117 (for n_envs == 1 identical return structure; batched arrays otherwise)."""
    observations, rewards, actions, infos = [], [], [], []
    obs = env.reset()
    observations.append(obs)
    while True:
        action = agent.get_action(obs)
        obs, reward, done, info = env.step(action)
        observations.append(obs); actions.append(action); rewards.append(reward); infos.append(info)
        if np.all(done):
            break
    return {"observations": observations, "actions": actions, "rewards": rewards, "infos": infos}
