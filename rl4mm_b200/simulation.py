"""Mirror of ``rl4mm/simulation`` (OrderbookSimulator, HistoricalOrderGenerator, OrderGenerator) and the
device-resident replacement of ``rl4mm/database`` for this path (:class:`DeviceDatabase`)."""
from __future__ import annotations

import abc
from datetime import datetime, timedelta
from typing import Dict, List, Optional

import numpy as np

from . import abi
from .orderbook import Exchange, FilledOrders, LimitOrder, MarketOrder, Order, Orderbook, _DIR
from .packing import PackedStream, RawMessages, compress_order_dict, pack_lobster, pack_merged, read_lobster_book_rows, read_lobster_messages


class DeviceDatabase:
    """Replaces ``HistoricalDatabase`` (rl4mm/database/HistoricalDatabase.py) for the hot path: packed ticker-days that
    are uploaded to HBM once instead of being queried from Postgres per episode / per step."""

    def __init__(self):
        self.streams: List[PackedStream] = []
        self.dates: List[datetime] = []
        self.tickers: List[str] = []

    def add_stream(self, ticker: str, trading_date: datetime, stream: PackedStream) -> int:
        self.streams.append(stream)
        self.dates.append(datetime.combine(trading_date.date(), datetime.min.time()))
        self.tickers.append(ticker)
        return len(self.streams) - 1

    def add_lobster_files(self, ticker: str, trading_date: datetime, message_csv, orderbook_csv, n_levels: int, **kw) -> int:
        s = pack_lobster(message_csv, orderbook_csv, n_levels, **kw)
        s.ticker, s.date = ticker, trading_date.strftime("%Y-%m-%d")
        return self.add_stream(ticker, trading_date, s)

    def add_merged_lobster_files(self, ticker: str, trading_date: datetime, message_csv, orderbook_csv, n_levels: int,
                                 extra_generators: Dict[str, RawMessages], **kw) -> int:
        """The reference's ``order_generators=[historical, ...]`` (OrderbookSimulator.py:24-53,74-75): the LOBSTER files plus
        the messages of further generators, merged at pack time with the reference's comparison
        (``_compress_order_dict``, :137-148) into one device-resident stream."""
        t, ty, oid, sz, pr, di = read_lobster_messages(message_csv, kw.pop("max_rows", None))
        sources = {"historical": RawMessages(t, ty, oid, sz, pr, di)}
        assert "historical" not in extra_generators
        sources.update(extra_generators)
        s = pack_merged(sources, lambda idx: read_lobster_book_rows(orderbook_csv, idx, n_levels), n_levels, **kw)
        s.ticker, s.date = ticker, trading_date.strftime("%Y-%m-%d")
        return self.add_stream(ticker, trading_date, s)

    def has_day(self, ticker: str, day: datetime) -> bool:
        """utils.daterange_in_db for one ticker-day (rl4mm/utils/utils.py:65-73)."""
        day = datetime.combine(day.date(), datetime.min.time())
        return any(t == ticker and d == day for t, d in zip(self.tickers, self.dates))

    def populate_from_archives(self, path_to_lobster_data, **kw) -> List[int]:
        """LOBSTER month archives (``*.7z``) of a folder, oldest first (run_populate_database_from_zipped.py:50-109); see
        ``rl4mm_b200.archives.populate_from_archives``."""
        from .archives import populate_from_archives

        return populate_from_archives(self, path_to_lobster_data, **kw)

    def stream_id(self, ticker: str, day: datetime) -> int:
        day = datetime.combine(day.date(), datetime.min.time())
        for i, (t, d) in enumerate(zip(self.tickers, self.dates)):
            if t == ticker and d == day:
                return i
        raise KeyError(f"no data for {ticker} on {day.date()}")

    def step_of(self, sid: int, t: datetime) -> int:
        s = self.streams[sid]
        us = (t - self.dates[sid]) // timedelta(microseconds=1) - s.t0_us
        if us % s.step_us:
            raise ValueError(f"{t} is not on the {s.step_us} us step grid")
        return us // s.step_us

    def time_of(self, sid: int, step: int) -> datetime:
        s = self.streams[sid]
        return self.dates[sid] + timedelta(microseconds=s.t0_us + step * s.step_us)


class OrderGenerator(metaclass=abc.ABCMeta):
    @property
    @abc.abstractmethod
    def name(self):
        pass


class HistoricalOrderGenerator(OrderGenerator):
    """rl4mm/simulation/HistoricalOrderGenerator.py -- here only a marker: the messages of every step are read by
    the kernel straight from the packed stream (CSR offsets), not materialised as Python Order objects."""

    name = "historical"

    def __init__(self, ticker: str = "MSFT", database: DeviceDatabase = None, preload_orders: bool = True):
        self.ticker, self.database, self.preload_orders = ticker, database, preload_orders
        self.exchange_name = "NASDAQ"


class PackedOrderGenerator(OrderGenerator):
    """A further OrderGenerator (rl4mm/simulation/OrderGenerator.py:9-21) next to the historical one.  Its messages were merged
    into the device-resident stream at pack time (``DeviceDatabase.add_merged_lobster_files``); the object is the name the
    simulator checks against ``PackedStream.generators``."""

    def __init__(self, name: str):
        self._name = name

    @property
    def name(self):
        return self._name


class OrderbookSimulator:
    """rl4mm/simulation/OrderbookSimulator.py:23-188 for one book (env 0 of its own LobSim, or a view of one env of a
    batched LobSim)."""

    _compress_order_dict = staticmethod(compress_order_dict)   # OrderbookSimulator.py:137-148 (the device path merges at pack time)

    def __init__(self, ticker: str = "MSFT", exchange: Exchange = None, order_generators=None, n_levels: int = 50,
                 database: DeviceDatabase = None, preload_orders: bool = True,
                 episode_length: timedelta = timedelta(minutes=30), warm_up: timedelta = timedelta(seconds=0),
                 outer_levels: int = 20, *, step_size: timedelta = timedelta(seconds=0.1), device: int = 0, **capacity):
        assert database is not None, "a DeviceDatabase with the packed stream(s) is required"
        self.ticker, self.n_levels, self.database = ticker, n_levels, database
        self.preload_orders, self.episode_length, self.warm_up, self.outer_levels = preload_orders, episode_length, warm_up, outer_levels
        self.step_size = step_size
        if exchange is None or exchange.sim.cfg.n_levels != n_levels or exchange.sim.cfg.outer_levels != outer_levels \
                or exchange.sim.cfg.fill_log_capacity == 0:
            from .device import LobSim

            cfg = abi.default_cfg(n_envs=1, n_levels=n_levels, outer_levels=outer_levels, fill_log_capacity=4096,
                                  step_us=step_size // timedelta(microseconds=1), **capacity)
            exchange = Exchange(ticker, sim=LobSim(cfg, device))
        self.exchange = exchange
        self.sim, self.env = exchange.sim, exchange.env
        for i, s in enumerate(database.streams):
            self.sim.load_stream(i, s)
        self.order_generators = {gen.name: gen for gen in (order_generators or [HistoricalOrderGenerator(ticker, database, preload_orders)])}
        for s in database.streams:                          # several generators: their messages must be IN the packed streams
            missing = set(self.order_generators) - set(s.generators)
            if missing:
                raise ValueError(f"order generators {sorted(missing)} are not part of the packed stream {s.ticker} {s.date} "
                                 f"(it holds {list(s.generators)}): pack with DeviceDatabase.add_merged_lobster_files")
        self.now_is: datetime = datetime(2000, 1, 1)
        self._sid = 0

    def reset_episode(self, start_date: datetime, start_book: Optional[Orderbook] = None):
        assert start_date.microsecond == 0, "Episodes must be started on the second."
        self._sid = self.database.stream_id(self.ticker, start_date)
        step = self.database.step_of(self._sid, start_date)
        self.exchange.use_stream_ids(self.database.streams[self._sid].ext_ids)
        self.sim.reset_book(self._sid, step, env_ids=[self.env])
        st = self.sim.state(self.env, 1)[0]
        assert not st["err"] & abi.ERR_NO_SNAPSHOT, f"There is no data before the episode start time: {start_date}"
        if start_book is not None:
            self.exchange.central_orderbook = start_book
        self.now_is = start_date
        return self.exchange.central_orderbook

    def forward_step(self, until: datetime, internal_orders: Optional[List[Order]] = None) -> FilledOrders:
        assert until > self.now_is, (f"The current time is {self.now_is.time()}, but we are trying to step forward in "
                                     f"time until {until.time()}!")
        filled = FilledOrders()
        for order in internal_orders or []:
            f = self.exchange.process_order(order)
            if f:
                filled.internal += f.internal
                filled.external += f.external
        n = self.database.step_of(self._sid, until) - self.database.step_of(self._sid, self.now_is)
        if self.sim.n_envs == 1:
            self.sim.forward_step(n)
        else:
            raise NotImplementedError("forward_step on a view of a batched LobSim: use the env API")
        for f in self.sim.fills(self.env):
            ref = int(f["ref"])
            is_agent = bool(ref & abi.REF_AGENT)
            if f["is_market"]:
                o = MarketOrder(until, _DIR[int(f["direction"])], self.ticker, None, None, False, int(f["volume"]), int(f["price"]))
            else:
                o = LimitOrder(None, _DIR[int(f["direction"])], self.ticker, -1 if ref == 0 else self.exchange._iid_of_ref.get(ref),
                               None if (is_agent or ref == 0) else self.exchange._ext_of_ref(ref),
                               not is_agent, int(f["price"]), int(f["volume"]))
            (filled.internal if f["list"] == 0 else filled.external).append(o)
        st = self.sim.state(self.env, 1)[0]
        if st["err"] & abi.ERR_EMPTY_BOOK:
            from .orderbook import EmptyOrderbookError

            raise EmptyOrderbookError("Trying take liquidity from an empty side of the book.")
        self.now_is = until
        return filled

    def book_depth(self, depth: int, orders: bool = False, agent: bool = False, out=None, stream=None):
        """L2 depth of EVERY env of the underlying LobSim (``LobSim.book_depth``): torch CUDA tensors [n_envs, 2, depth],
        batched and not squeezed, also when n_envs == 1 or this simulator is a view of one env (index with ``self.env``)."""
        return self.sim.book_depth(depth, orders=orders, agent=agent, out=out, stream=stream)

    def agent_orders(self, max_orders=None, queue: bool = True, out=None, stream=None):
        """The agent's orders and queue positions in EVERY env of the underlying LobSim (``LobSim.agent_orders``), batched
        and not squeezed, also when n_envs == 1 or this simulator is a view of one env (index with ``self.env``)."""
        return self.sim.agent_orders(max_orders=max_orders, queue=queue, out=out, stream=stream)

    def book_l3(self, max_entries=None, out=None, stream=None):
        """The L3 book of EVERY env of the underlying LobSim (``LobSim.book_l3``): count [n_envs, 2], entries
        [n_envs, 2, max_entries, 4], batched and not squeezed, also when n_envs == 1 or this simulator is a view of one env
        (index with ``self.env``)."""
        return self.sim.book_l3(max_entries=max_entries, out=out, stream=stream)

    @property
    def min_buy_price(self) -> int:
        return int(self.sim.state(self.env, 1)[0]["min_buy_price"])

    @property
    def max_sell_price(self) -> int:
        return int(self.sim.state(self.env, 1)[0]["max_sell_price"])
