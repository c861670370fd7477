"""TEST INFRASTRUCTURE ONLY -- import shims that let the *unmodified* reference (a checkout of the original rl4mm
project, located by the environment variable ``RL4MM_REFERENCE``) run so that golden vectors can be generated from it
(see ``oracle/gen_golden.py``).

Nothing in the product path (``rl4mm_b200/``), ``bench.py`` or the ``-m gpu`` tests imports this module: the reference
is not part of this repository.  The vectors this module helps to produce are committed under ``tests/golden/``.

What is shimmed (SURVEY.md App. B):
  * ``numpy.infty`` (removed in numpy 2; evaluated eagerly at rl4mm/orderbook/Exchange.py:154,
    rl4mm/orderbook/models.py:77, rl4mm/simulation/OrderbookSimulator.py:51-53);
  * stub modules for sqlalchemy / gym / ray / pandas_market_calendars / plotly / mypy_extensions /
    matplotlib / seaborn / numpyencoder / tqdm-free imports, none of which is on the hot path;
  * an in-memory stand-in for ``rl4mm.database.HistoricalDatabase`` that restates the loader semantics of
    rl4mm/database/database_population_helpers.py:116-160 (type map, direction flip, microsecond timestamps),
    :45-62,139-148 (snapshot alignment), :163-181 (id string => lexicographic tie order) and the queries of
    rl4mm/database/HistoricalDatabase.py:46-62,103-119.
"""
from __future__ import annotations

import os
import sys
import types
from datetime import datetime, timedelta
from pathlib import Path

import numpy as np
import pandas as pd

REFERENCE_ROOT = Path(os.environ["RL4MM_REFERENCE"]) if os.environ.get("RL4MM_REFERENCE") else None
_INSTALLED = False


def _module(name: str, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules[name] = mod
    return mod


class _Box:
    """Minimal gym.spaces.Box (used at rl4mm/gym/HistoricalOrderbookEnvironment.py:88-94,125-135)."""

    def __init__(self, low, high, shape=None, dtype=None):
        if shape is not None:
            low = np.full(shape, low, dtype=dtype)
            high = np.full(shape, high, dtype=dtype)
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = dtype
        self._rng = np.random.default_rng()

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)

    def sample(self):
        return self._rng.uniform(self.low, self.high)


class _Env:
    def __init__(self):
        pass


def install() -> None:
    """Register the stubs and put the reference on ``sys.path``.  Idempotent."""
    global _INSTALLED
    if _INSTALLED:
        return
    if REFERENCE_ROOT is None or not (REFERENCE_ROOT / "rl4mm").is_dir():
        raise RuntimeError("set RL4MM_REFERENCE to a checkout of the original rl4mm project")
    if not hasattr(np, "infty"):
        np.infty = np.inf  # noqa: NPY201

    anything = lambda *a, **k: None  # noqa: E731

    class _Base:
        metadata = types.SimpleNamespace(create_all=anything)

    sa = _module(
        "sqlalchemy", create_engine=anything, Column=anything, DateTime=anything, Integer=anything, JSON=anything,
        String=anything,
    )
    sa.engine = _module("sqlalchemy.engine")
    sa.engine.base = _module("sqlalchemy.engine.base", Engine=object)
    sa.orm = _module("sqlalchemy.orm", sessionmaker=anything)
    sa.ext = _module("sqlalchemy.ext")
    sa.ext.declarative = _module("sqlalchemy.ext.declarative", declarative_base=lambda: _Base)
    sa.exc = _module("sqlalchemy.exc", IntegrityError=Exception)
    _module("mypy_extensions", TypedDict=dict)
    px = _module("plotly")
    px.express = _module("plotly.express")
    _module("pandas_market_calendars", get_calendar=anything)
    ray = _module("ray")
    ray.tune = _module("ray.tune")
    ray.tune.logger = _module("ray.tune.logger", UnifiedLogger=object)
    gym = _module("gym", Env=_Env)
    gym.spaces = _module("gym.spaces", Box=_Box)
    gym.utils = _module("gym.utils")
    gym.utils.seeding = _module("gym.utils.seeding", np_random=lambda seed=None: (np.random.default_rng(seed), seed))
    gym.utils.seeding_mod = gym.utils.seeding
    gym.envs = _module("gym.envs")
    gym.envs.registration = _module("gym.envs.registration", EnvSpec=lambda **k: types.SimpleNamespace(**k))
    # plotting / JSON helpers imported at module level by rl4mm/gym/utils.py:8-15 (evaluation path); never called here
    mpl = _module("matplotlib")
    mpl.pyplot = _module("matplotlib.pyplot")
    _module("seaborn")
    import json as _json

    class _NumpyEncoder(_json.JSONEncoder):
        def default(self, o):
            return o.tolist() if isinstance(o, (np.ndarray, np.generic)) else super().default(o)

    _module("numpyencoder", NumpyEncoder=_NumpyEncoder)
    sys.path.insert(0, str(REFERENCE_ROOT))
    import rl4mm.gym.HistoricalOrderbookEnvironment as hoe  # noqa: E402

    # the NASDAQ calendar is only used to pick the trading day (HOE.py:348-351)
    hoe.get_next_trading_dt = lambda ts: datetime.combine(pd.Timestamp(ts).date(), datetime.min.time()) + timedelta(
        hours=9, minutes=30
    )
    _INSTALLED = True


# ---------------------------------------------------------------------------------------------------------------------
#  in-memory HistoricalDatabase stand-in
# ---------------------------------------------------------------------------------------------------------------------

TYPE_MAP = {1: "limit", 2: "cancellation", 3: "deletion", 4: "market", 5: "market_hidden", 6: "cross_trade",
            7: "trading_halt"}  # database_population_helpers.py:151-160


def book_columns(n_levels: int):
    """Column order of a LOBSTER orderbook row -- rl4mm/orderbook/helpers.py:52-55."""
    cols = []
    for i in range(n_levels):
        cols += [f"sell_price_{i}", f"sell_volume_{i}", f"buy_price_{i}", f"buy_volume_{i}"]
    return cols


def parse_lobster_time_ns(text: str) -> int:
    """LOBSTER seconds-after-midnight decimal string -> integer nanoseconds (exact, no float)."""
    if "." in text:
        sec, frac = text.split(".")
    else:
        sec, frac = text, ""
    frac = (frac + "000000000")[:9]
    return int(sec) * 1_000_000_000 + int(frac)


class InMemoryDatabase:
    """Duck-types rl4mm.database.HistoricalDatabase for OrderbookSimulator / HistoricalOrderGenerator.

    ``tie_order="reference"`` orders same-microsecond messages by the *string* id
    (HistoricalDatabase.py:111 ``order_by(timestamp, id)``, id from database_population_helpers.py:163-164);
    ``tie_order="file"`` keeps file order.
    """

    exchange = "NASDAQ"

    def __init__(self, message_csv, book_csv, ticker: str, trading_date: datetime, n_levels: int,
                 snapshot_freq=None, max_rows: int | None = None, tie_order: str = "reference"):
        self.ticker, self.n_levels = ticker, n_levels
        rows = []
        with open(message_csv) as f:
            for i, line in enumerate(f):
                if max_rows is not None and i >= max_rows:
                    break
                p = line.strip().split(",")
                rows.append((parse_lobster_time_ns(p[0]), int(p[1]), int(p[2]), int(p[3]), int(p[4]), int(p[5])))
        t_ns = np.array([r[0] for r in rows], dtype=np.int64)
        mtype = [TYPE_MAP[r[1]] for r in rows]
        direction = []
        for r, mt in zip(rows, mtype):  # database_population_helpers.py:132-136
            if mt == "market":
                direction.append("sell" if r[5] == 1 else "buy")
            else:
                direction.append("buy" if r[5] == 1 else "sell")
        day = datetime.combine(pd.Timestamp(trading_date).date(), datetime.min.time())
        date_str = day.strftime("%Y-%m-%d")
        # SQL DateTime => python datetime => microsecond resolution (truncation of the ns part)
        ts = [day + timedelta(microseconds=int(t // 1000)) for t in t_ns]
        ids = [f"{snapshot_freq}_L{str(n_levels).zfill(3)}_NASDAQ_{ticker}_{date_str}_{i}" for i in range(len(rows))]
        self.messages = pd.DataFrame(
            dict(
                id=ids, timestamp=pd.Series(ts, dtype="datetime64[us]"), exchange="NASDAQ", ticker=ticker,
                direction=direction, volume=[r[3] for r in rows], price=[r[4] for r in rows],
                external_id=[r[2] for r in rows], message_type=mtype,
            )
        )
        self.messages["_row"] = np.arange(len(rows))
        if tie_order == "reference":
            self.messages = self.messages.sort_values(["timestamp", "id"], kind="stable").reset_index(drop=True)
        elif tie_order != "file":
            raise ValueError(tie_order)
        self._ts_py = [t.to_pydatetime() for t in self.messages.timestamp]
        books = np.loadtxt(book_csv, delimiter=",", dtype=np.int64, max_rows=len(rows))
        self._cols = book_columns(n_levels)
        # snapshot rows: database_population_helpers.py:45-62,139-148
        if snapshot_freq is None:
            keep = np.arange(len(rows))
            snap_ts = [day + timedelta(microseconds=int(t // 1000)) for t in t_ns]
        else:
            assert snapshot_freq == "S"
            first = -(-t_ns[0] // 1_000_000_000)
            last = -(-t_ns[-1] // 1_000_000_000)
            keep, seen = [], set()
            for sec in range(int(first), int(last) + 1):
                idx = int(np.searchsorted(t_ns, sec * 1_000_000_000, side="right")) - 1
                if idx >= 0 and idx not in seen:
                    seen.add(idx)
                    keep.append(idx)
            keep = np.array(keep, dtype=np.int64)
            snap_ts = [day + timedelta(microseconds=int(t_ns[i] // 1000)) for i in keep]
        # get_last_snapshot orders by (timestamp desc, id desc), get_next_snapshot by (timestamp asc, id asc)
        # with the *string* id (HistoricalDatabase.py:52,70) => sort snapshot rows by (timestamp, id string).
        snap_us = [(t - day) // timedelta(microseconds=1) for t in snap_ts]
        order = sorted(range(len(keep)), key=lambda j: (snap_us[j], ids[int(keep[j])]))
        self._snap_rows = books[keep][order]
        self._snap_ts = [snap_ts[j] for j in order]
        self._snap_key = np.array([snap_us[j] for j in order], dtype=np.int64)
        self._day = day

    def _us(self, t: datetime) -> int:
        return (pd.Timestamp(t).to_pydatetime() - self._day) // timedelta(microseconds=1)

    def get_messages(self, start_date, end_date, ticker):
        m = self.messages
        sel = m[(m.timestamp > pd.Timestamp(start_date)) & (m.timestamp <= pd.Timestamp(end_date))]
        if len(sel) == 0:
            return pd.DataFrame()
        out = sel.drop(columns=["_row"]).reset_index(drop=True)
        out["timestamp"] = [t.to_pydatetime() for t in out.timestamp]
        return out

    def _series(self, i):
        return pd.Series(dict(zip(self._cols, (int(v) for v in self._snap_rows[i]))), name=self._snap_ts[i])

    def get_last_snapshot(self, timestamp, ticker):
        i = int(np.searchsorted(self._snap_key, self._us(timestamp), side="right")) - 1
        return pd.DataFrame() if i < 0 else self._series(i)

    def get_next_snapshot(self, timestamp, ticker):
        i = int(np.searchsorted(self._snap_key, self._us(timestamp), side="left"))
        return pd.DataFrame() if i >= len(self._snap_key) else self._series(i)


def import_eval_utils():
    """Import rl4mm/gym/utils.py (generate_trajectory, episode summary dict).  Its module-level default argument
    `database=HistoricalDatabase()` (utils.py:42) opens a Postgres engine at import time; neutralise the constructor
    for the duration of the import only."""
    install()
    import rl4mm.database.HistoricalDatabase as hd

    orig = hd.HistoricalDatabase.__init__
    hd.HistoricalDatabase.__init__ = lambda self, *a, **k: None
    try:
        import rl4mm.gym.utils as utils
    finally:
        hd.HistoricalDatabase.__init__ = orig
    return utils
