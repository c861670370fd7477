"""TEST INFRASTRUCTURE: generate the golden vectors under tests/golden/ by running the UNMODIFIED reference
(a checkout of the original rl4mm project, imported through oracle/refshim.py).

    RL4MM_REFERENCE=<rl4mm checkout> python -m oracle.gen_golden            # rewrites tests/golden/*.json.gz

The reference cannot travel to the GPU box, the vectors can.  tests/test_oracle_golden.py pins the C oracle against
them (CPU), tests/test_gpu_parity.py pins the CUDA path against them and against the oracle (GPU).
"""
from __future__ import annotations

import gzip
import json
import sys
from datetime import datetime, timedelta
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import refshim  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"
FIXTURE_DIR = Path(refshim.REFERENCE_ROOT or "") / "test_data"     # refshim.install() refuses to run without the reference
MSG_CSV = FIXTURE_DIR / "MSFT_2012-06-21_34200000_37800000_message_50.csv"
BOOK_CSV = FIXTURE_DIR / "MSFT_2012-06-21_34200000_37800000_orderbook_50.csv"
DAY = datetime(2012, 6, 21)


def save(name: str, obj) -> None:
    GOLDEN.mkdir(parents=True, exist_ok=True)
    with gzip.GzipFile(GOLDEN / name, "wb", mtime=0) as f:
        f.write(json.dumps(obj, separators=(",", ":")).encode())
    print("wrote", name, (GOLDEN / name).stat().st_size, "bytes")


def dump_book(orderbook):
    """Canonical L3 dump: per side (buy best-first, sell best-first) [price, volume, kind, ext_id];
    kind 0 = snapshot aggregate (internal_id -1), 1 = external order, 2 = agent order."""
    out = []
    for direction in ("buy", "sell"):
        side = getattr(orderbook, direction)
        prices = list(reversed(side)) if direction == "buy" else list(side)
        rows = []
        for p in prices:
            for o in side[p]:
                if not o.is_external:
                    rows.append([int(p), int(o.volume), 2, 0])
                elif o.internal_id == -1:
                    rows.append([int(p), int(o.volume), 0, 0])
                else:
                    rows.append([int(p), int(o.volume), 1, int(o.external_id)])
        out.append(rows)
    return out


def dump_fills(filled):
    from rl4mm.orderbook.models import MarketOrder

    out = []
    for lst, orders in ((0, filled.internal), (1, filled.external)):
        for o in orders:
            out.append([lst, 0 if o.direction == "buy" else 1, int(o.price), int(o.volume), int(isinstance(o, MarketOrder))])
    return out  # NOTE: internal and external lists are separate in the reference; order is kept within each list


def make_db(snapshot_freq="S", tie_order="reference"):
    return refshim.InMemoryDatabase(MSG_CSV, BOOK_CSV, "MSFT", DAY, 50, snapshot_freq, 1000, tie_order)


def make_sim(db, outer_levels=20, preload=False, episode_length=None, warm_up=timedelta(0)):
    from rl4mm.orderbook.Exchange import Exchange
    from rl4mm.simulation.HistoricalOrderGenerator import HistoricalOrderGenerator
    from rl4mm.simulation.OrderbookSimulator import OrderbookSimulator

    gen = HistoricalOrderGenerator("MSFT", db, preload_orders=preload)
    return OrderbookSimulator("MSFT", Exchange("MSFT"), [gen], 50, db, preload_orders=preload,
                              episode_length=episode_length, warm_up=warm_up, outer_levels=outer_levels)


# ---------------------------------------------------------------------------------------------------------------------
def golden_fixture_replay():
    """G1: OrderbookSimulator.forward_step over the MSFT fixture in 0.1 s steps; L3 book + fills after every step."""
    cases = []
    for outer_levels in (20, 48):
        for tie in ("reference", "file"):
            sim = make_sim(make_db("S", tie), outer_levels)
            start = DAY + timedelta(hours=10)
            sim.reset_episode(start)
            steps = [dict(book=dump_book(sim.exchange.central_orderbook), fills=[],
                          min_buy=int(sim.min_buy_price), max_sell=int(sim.max_sell_price))]
            now = start
            for _ in range(27):
                now += timedelta(seconds=0.1)
                filled = sim.forward_step(now)
                steps.append(dict(book=dump_book(sim.exchange.central_orderbook), fills=dump_fills(filled),
                                  min_buy=int(sim.min_buy_price), max_sell=int(sim.max_sell_price)))
            cases.append(dict(outer_levels=outer_levels, tie_order=tie, start_seconds=36000, steps=steps))
    save("fixture_replay.json.gz", cases)


# ---------------------------------------------------------------------------------------------------------------------
def feature_specs():
    """(reference constructor, abi description) pairs for a feature set with windows that fit the 3 s fixture."""
    from rl4mm.features import Features as F

    td = timedelta
    return [
        (lambda: F.Spread(), dict(kind="SPREAD", lookback=0, update_us=100000, min=0, max=5000)),
        (lambda: F.BookImbalance(), dict(kind="BOOK_IMBALANCE", lookback=0, update_us=100000, min=-1, max=1)),
        (lambda: F.PriceMove(name="pm1", update_frequency=td(seconds=0.1), lookback_periods=1),
         dict(kind="PRICE_MOVE", lookback=1, update_us=100000, min=-10000, max=10000)),
        (lambda: F.PriceMove(name="pm3", update_frequency=td(seconds=0.2), lookback_periods=3),
         dict(kind="PRICE_MOVE", lookback=3, update_us=200000, min=-10000, max=10000)),
        (lambda: F.PriceRange(update_frequency=td(seconds=0.1), lookback_periods=3),
         dict(kind="PRICE_RANGE", lookback=3, update_us=100000, min=0, max=10000)),
        (lambda: F.Volatility(name="v4", update_frequency=td(seconds=0.1), lookback_periods=4, max_value=1e-9),
         dict(kind="VOLATILITY", lookback=4, update_us=100000, min=0, max=1e-9)),
        (lambda: F.Price(update_frequency=td(seconds=0.5)),
         dict(kind="PRICE", lookback=0, update_us=500000, min=0, max=100000000)),
        (lambda: F.TradeDirectionImbalance(update_frequency=td(seconds=0.1), lookback_periods=5),
         dict(kind="TRADE_DIR_IMBALANCE", lookback=5, update_us=100000, min=-1, max=1, iparam=0)),
        (lambda: F.TradeVolumeImbalance(update_frequency=td(seconds=0.1), lookback_periods=5, track_internal=True),
         dict(kind="TRADE_VOL_IMBALANCE", lookback=5, update_us=100000, min=-1, max=1, iparam=1)),
        (lambda: F.Inventory(), dict(kind="INVENTORY", lookback=0, update_us=100000, min=-1000000, max=1000000)),
        (lambda: F.EpisodeProportion(update_frequency=td(seconds=0.1), episode_length=td(seconds=1.5)),
         dict(kind="EPISODE_PROPORTION", lookback=0, update_us=100000, min=0, max=1, dparam=0.1 / 1.5)),
        (lambda: F.TimeOfDay(update_frequency=td(seconds=1), n_buckets=10),
         dict(kind="TIME_OF_DAY", lookback=0, update_us=1000000, min=0, max=9, iparam=10)),
        # the two features of the reference's own env test (testHistoricalOrderbookEnvironment.py:43); 1 s windows
        (lambda: F.PriceMove(lookback_periods=1),
         dict(kind="PRICE_MOVE", lookback=1, update_us=1000000, min=-10000, max=10000)),
        (lambda: F.PriceRange(lookback_periods=1),
         dict(kind="PRICE_RANGE", lookback=1, update_us=1000000, min=0, max=10000)),
        # index 14: AmihudLambda, window (4 + 1) * 2 * 0.1 s = 1 s
        (lambda: F.AmihudLambda(update_frequency=td(seconds=0.1), lookback_periods=4, slowing_factor=2, max_value=1e-3),
         dict(kind="AMIHUD_LAMBDA", lookback=10, update_us=100000, min=0, max=1e-3, iparam=2)),
        # indices 15-19: rolling z-score normalisation (Features.py:67-74), short histories so that eviction happens
        (lambda: F.Spread(normalisation_on=True, max_norm_len=6),
         dict(kind="SPREAD", lookback=0, update_us=100000, min=0, max=5000, norm_len=6)),
        (lambda: F.PriceMove(name="pmn", update_frequency=td(seconds=0.1), lookback_periods=2, normalisation_on=True, max_norm_len=5),
         dict(kind="PRICE_MOVE", lookback=2, update_us=100000, min=-10000, max=10000, norm_len=5)),
        (lambda: F.Volatility(name="vn", update_frequency=td(seconds=0.1), lookback_periods=3, normalisation_on=True, max_norm_len=100),
         dict(kind="VOLATILITY", lookback=3, update_us=100000, min=0, max=1.0, norm_len=100)),
        (lambda: F.Inventory(normalisation_on=True, max_norm_len=7),
         dict(kind="INVENTORY", lookback=0, update_us=100000, min=-1000000, max=1000000, norm_len=7)),
        (lambda: F.TradeVolumeImbalance(update_frequency=td(seconds=0.1), lookback_periods=10, normalisation_on=True, max_norm_len=1000),
         dict(kind="TRADE_VOL_IMBALANCE", lookback=10, update_us=100000, min=-1, max=1, iparam=0, norm_len=1000)),
        # indices 20-22: windows that stay (nearly) constant at a large, non-integer magnitude -- scipy's "std <= |eps * mean|
        # -> NaN" rule and numpy's rounding in the noise-dominated window [p + 1e-06, p, p, ...]
        (lambda: F.Price(name="pn4", update_frequency=td(seconds=0.1), normalisation_on=True, max_norm_len=4),
         dict(kind="PRICE", lookback=0, update_us=100000, min=0, max=100000000, norm_len=4)),
        (lambda: F.Price(name="pn300", update_frequency=td(seconds=0.1), normalisation_on=True, max_norm_len=300),
         dict(kind="PRICE", lookback=0, update_us=100000, min=0, max=100000000, norm_len=300)),
        (lambda: F.PriceRange(name="prn", update_frequency=td(seconds=0.1), lookback_periods=10, normalisation_on=True, max_norm_len=9),
         dict(kind="PRICE_RANGE", lookback=10, update_us=100000, min=0, max=10000, norm_len=9)),
    ]


def run_env_case(name, actions, env_kwargs, reward_step, reward_term, features=None, episode_seconds=1.5,
                 start_seconds=36001.0, n_episodes=1, outer_levels=20, portfolio=None, step_hook=None):
    from rl4mm.features.Features import Portfolio
    from rl4mm.gym.HistoricalOrderbookEnvironment import HistoricalOrderbookEnvironment
    from rl4mm.rewards.RewardFunctions import InventoryAdjustedPnL, PnL

    def reward(spec):
        from rl4mm.rewards.RewardFunctions import RollingSharpe

        if spec[0] == "PnL":
            return PnL()
        if spec[0] == "RS":
            return RollingSharpe(max_window_size=spec[1], min_window_size=spec[2])
        return InventoryAdjustedPnL(inventory_aversion=spec[1], asymmetrically_dampened=spec[2])

    specs = feature_specs()[:14] if features is None else [feature_specs()[i] for i in features]
    feats = [mk() for mk, _ in specs]
    max_window = max(f.window_size for f in feats)
    episode_length = timedelta(seconds=episode_seconds)
    db = make_db("S", "reference")
    sim = make_sim(db, outer_levels, preload=True, episode_length=episode_length, warm_up=max_window)
    start_td = timedelta(seconds=start_seconds)
    env = HistoricalOrderbookEnvironment(
        features=feats, ticker="MSFT", step_size=timedelta(seconds=0.1), episode_length=episode_length,
        initial_portfolio=Portfolio(*portfolio) if portfolio else None, min_date=DAY, max_date=DAY,
        min_start_timedelta=start_td, max_end_timedelta=start_td + episode_length, simulator=sim,
        per_step_reward_function=reward(reward_step), terminal_reward_function=reward(reward_term), n_levels=50,
        **env_kwargs,
    )
    episodes = []
    k = 0
    for _ in range(n_episodes):
        obs0 = env.reset()
        ep = dict(reset_obs=[float(x) for x in obs0], reset_book=dump_book(env.central_orderbook),
                  reset_inventory=int(env.state.portfolio.inventory), reset_cash=float(env.state.portfolio.cash),
                  steps=[])
        while True:
            a = actions[k % len(actions)]
            k += 1
            orders = None
            obs, r, done, _ = env.step(np.array(a, dtype=float))
            ep["steps"].append(dict(
                action=[float(x) for x in a], obs=[float(x) for x in obs], reward=float(r), done=bool(done),
                inventory=int(env.state.portfolio.inventory), cash=float(env.state.portfolio.cash),
                price=float(env.state.price), book=dump_book(env.central_orderbook),
                agent_book=dump_book(env.internal_orderbook), fills=dump_fills(env.state.filled_orders),
            ))
            if step_hook is not None:
                step_hook(env, ep["steps"][-1])
            if done:
                break
        episodes.append(ep)
    return dict(
        name=name, env_kwargs={k_: v for k_, v in env_kwargs.items()}, reward_step=reward_step, reward_term=reward_term,
        features=[d for _, d in specs], episode_steps=int(round(episode_seconds * 10)),
        warmup_steps=int(max_window / timedelta(seconds=0.1)), start_seconds=start_seconds, outer_levels=outer_levels,
        portfolio=list(portfolio) if portfolio else [0, 1000], episodes=episodes,
    )


def golden_env_episodes():
    """G2: HistoricalOrderbookEnvironment reset/step traces on the MSFT fixture."""
    rng = np.random.default_rng(1234)
    rand4 = rng.uniform(0.0, 10.0, size=(64, 4)).tolist()
    rand5 = np.c_[rng.uniform(0.0, 10.0, size=(64, 4)), rng.uniform(0, 60, size=64)].tolist()
    rand2 = rng.uniform(0.0, 10.0, size=(64, 2)).tolist()
    cases = [
        run_env_case("fixed_1212_pnl", [[1, 2, 1, 2]], {}, ("PnL",), ("PnL",)),
        run_env_case("fixed_1111_default_rewards", [[1, 1, 1, 1]], {}, ("IA", 1e-4, False), ("IA", 0.1, False)),
        run_env_case("random_asym", rand4, {}, ("IA", 0.01, True), ("IA", 0.5, True), n_episodes=2),
        run_env_case("random_two_episodes_carryover", rand4[7:], {"inc_prev_action_in_obs": True}, ("PnL",),
                     ("IA", 0.1, False), n_episodes=3, start_seconds=36000.0 + 1.0, episode_seconds=1.0),
        run_env_case("enter_spread", rand4[20:], {"enter_spread": True}, ("PnL",), ("PnL",)),
        run_env_case("market_order_clearing", rand5,
                     {"market_order_clearing": True, "market_order_fraction_of_inventory": 0.3, "max_inventory": 60},
                     ("PnL",), ("PnL",), n_episodes=2),
        run_env_case("concentration", rand2, {"concentration": 10.0}, ("PnL",), ("PnL",)),
        run_env_case("quote_levels_3_8", rand4[30:], {"min_quote_level": 3, "max_quote_level": 8}, ("PnL",), ("PnL",)),
        run_env_case("float_cash", rand4[40:], {}, ("PnL",), ("PnL",), portfolio=(25, 1e12)),
        run_env_case("reference_test_features", [[1, 2, 1, 2]], {}, ("IA", 1e-4, False), ("IA", 0.1, False),
                     features=[9, 0, 12, 13], episode_seconds=1.0, start_seconds=36001.0),
        run_env_case("amihud_rolling_sharpe", rand4[50:], {}, ("RS", 6, 3), ("RS", 4, 2), features=[14, 9, 0, 7],
                     n_episodes=3, episode_seconds=1.0, start_seconds=36001.0, portfolio=(0, 10**10)),
        run_env_case("amihud_full", rand4[10:], {}, ("RS", 12, 5), ("PnL",), features=list(range(12)) + [14],
                     portfolio=(0, 10**10)),
        run_env_case("normalised_features", rand4[25:], {}, ("PnL",), ("PnL",), features=[15, 16, 17, 18, 19, 9],
                     n_episodes=2, episode_seconds=1.5, start_seconds=36001.0),
        run_env_case("normalised_constant_windows", [[1, 2, 1, 2]], {}, ("PnL",), ("PnL",), features=[20, 21, 22, 0],
                     n_episodes=2, episode_seconds=2.0, start_seconds=36000.0 + 1.0),
    ]
    save("env_episodes.json.gz", cases)


def golden_env_random():
    """G2b: the reference env on the MSFT fixture under RANDOM configurations (seeded): env kwargs, feature subsets, reward
    kinds, portfolios and actions are drawn at random, so that the pins are not limited to hand-picked cases."""
    rng = np.random.default_rng(2024)
    n_specs = len(feature_specs())
    cases = []
    for k in range(16):
        feats = sorted(set([int(rng.choice([12, 13, 14, 22]))] + [int(i) for i in rng.choice(n_specs, size=int(rng.integers(2, 9)), replace=False)]))
        conc = bool(rng.random() < 0.25)
        clearing = bool(rng.random() < 0.35)
        kw = {}
        if conc:
            kw["concentration"] = 10.0
        if clearing:
            kw.update(market_order_clearing=True, market_order_fraction_of_inventory=float(rng.choice([0.3, 1.0])), max_inventory=60)
        if rng.random() < 0.4:
            kw["enter_spread"] = True
        if rng.random() < 0.4:
            kw["inc_prev_action_in_obs"] = True
        if rng.random() < 0.5:
            lo = int(rng.integers(0, 3))
            kw.update(min_quote_level=lo, max_quote_level=lo + int(rng.choice([3, 5, 10])))
        ad = (2 if conc else 4)
        acts = rng.uniform(0.0, 10.0, size=(64, ad))
        acts[rng.random(acts.shape) < 0.05] = 0.0
        if clearing:
            acts = np.c_[acts, rng.uniform(0, 80, size=64)]

        def reward():
            r = int(rng.integers(0, 4))
            if r == 0:
                return ("PnL",)
            if r == 3:
                mx = int(rng.integers(3, 9))
                return ("RS", mx, int(rng.integers(2, mx + 1)))
            return ("IA", float(rng.choice([1e-4, 0.01, 0.5])), bool(r == 2))

        cases.append(run_env_case(
            f"random_{k}", acts.tolist(), kw, reward(), reward(), features=feats, n_episodes=int(rng.integers(1, 4)),
            episode_seconds=float(rng.choice([1.0, 1.5, 2.0])), start_seconds=36000.0 + 1.0,
            outer_levels=int(rng.choice([20, 48])), portfolio=(int(rng.choice([0, 0, 25, -40])), int(rng.choice([10**8, 10**10])))))
    save("env_random.json.gz", cases)


# ---------------------------------------------------------------------------------------------------------------------
def golden_beta_ladders():
    """G3: BetaOrderDistributor lot sizes (scipy.stats.beta.pdf + np.round half-to-even)."""
    from rl4mm.gym.action_interpretation.OrderDistributors import BetaOrderDistributor

    rng = np.random.default_rng(99)
    out = []
    for Q, vol, conc in ((10, 100, None), (5, 100, None), (8, 37, None), (16, 250, None), (10, 100, 10.0), (10, 100, 25.0)):
        dist = BetaOrderDistributor(Q, active_volume=vol, concentration=conc)
        n = 2 if conc is not None else 4
        acts = [list(map(float, a)) for a in rng.uniform(0, 10 if conc is None else conc, size=(150, n))]
        acts += [[float(i), float(j)] * (n // 2) for i in range(0, 11, 2) for j in range(0, 11, 2)] if conc is None else \
                [[float(i), float(j)] for i in range(0, 11, 2) for j in range(0, 11, 2)]
        rows = []
        for a in acts:
            d = dist.convert_action(np.array(a))
            rows.append(dict(action=a, buy=[int(x) for x in d["buy"]], sell=[int(x) for x in d["sell"]]))
        out.append(dict(quote_levels=Q, active_volume=vol, concentration=conc, cases=rows))
    save("beta_ladders.json.gz", out)


# ---------------------------------------------------------------------------------------------------------------------
def golden_exchange_fuzz():
    """G5: random order sequences (external + agent, unknown ids, over-size cancels, self-matches, volume-less
    deletions) through the reference Exchange; fills per order and the final L3 books."""

    from rl4mm.orderbook.Exchange import EmptyOrderbookError, Exchange
    from rl4mm.orderbook.models import Cancellation, Deletion, LimitOrder, MarketOrder

    rng = np.random.default_rng(7)
    ts = datetime(2012, 6, 21, 12)
    cases = []
    for case in range(120):
        ex = Exchange("MSFT")
        mid = 300000
        # snapshot aggregates on both sides (internal_id -1)
        init = []
        for k in range(1, 6):
            for direction, price in (("buy", mid - 100 * k), ("sell", mid + 100 * k)):
                if rng.random() < 0.8:
                    init.append(LimitOrder(ts, direction, "MSFT", -1, None, True, price, int(rng.integers(1, 9)) * 100))
        ex.central_orderbook = ex.get_initial_orderbook_from_orders(init)
        seq = []
        next_ext = 1
        live_ext = []     # (ext_id, direction, price)
        agent_live = []   # (internal_id, direction, price)
        dead = False
        for _ in range(int(rng.integers(30, 120))):
            u = rng.random()
            is_agent = rng.random() < 0.3
            direction = "buy" if rng.random() < 0.5 else "sell"
            price = int(mid + 100 * rng.integers(-7, 8))
            vol = int(rng.integers(1, 12)) * 50
            rec = None
            if u < 0.45:
                if is_agent:
                    order = LimitOrder(ts, direction, "MSFT", None, None, False, price, vol)
                    rec = dict(type=1, dir=direction, price=price, vol=vol, ext=False, ref=0)
                else:
                    order = LimitOrder(ts, direction, "MSFT", None, next_ext, True, price, vol)
                    rec = dict(type=1, dir=direction, price=price, vol=vol, ext=True, ref=next_ext)
                    live_ext.append((next_ext, direction, price))
                    next_ext += 1
            elif u < 0.60:
                order = MarketOrder(ts, direction, "MSFT", None, None if is_agent else next_ext, not is_agent, vol)
                rec = dict(type=4, dir=direction, price=0, vol=vol, ext=not is_agent, ref=0 if is_agent else next_ext)
                if not is_agent:
                    next_ext += 1
            else:
                ctype = Cancellation if u < 0.8 else Deletion
                t = 2 if u < 0.8 else 3
                if is_agent and agent_live:
                    iid, d_, p_ = agent_live[int(rng.integers(len(agent_live)))]
                    v = None if (t == 3 and rng.random() < 0.5) else vol
                    order = ctype(ts, d_, "MSFT", iid, None, False, p_, v)
                    rec = dict(type=t, dir=d_, price=p_, vol=0 if v is None else v, ext=False, ref=-1, agent_index=iid)
                else:
                    r = rng.random()
                    if live_ext and r < 0.7:
                        e, d_, p_ = live_ext[int(rng.integers(len(live_ext)))]
                        if rng.random() < 0.1:
                            p_ += 100  # wrong price level
                    else:
                        e, d_, p_ = int(10_000 + rng.integers(100)), direction, price  # unknown id => aggregates
                    v = vol
                    if t == 3 and r < 0.35 and live_ext:
                        v = None  # only for ids that exist (the reference asserts on aggregates)
                        # make sure the level's head is not an aggregate when the order is gone
                    order = ctype(ts, d_, "MSFT", None, e, True, p_, v)
                    rec = dict(type=t, dir=d_, price=p_, vol=0 if v is None else v, ext=True, ref=e)
            before_counter = ex.order_id_convertor.counter
            try:
                filled = ex.process_order(order)
            except EmptyOrderbookError:
                rec["raised"] = "EmptyOrderbookError"
                seq.append(rec)
                dead = True
                break
            except AssertionError:
                rec["raised"] = "AssertionError"
                seq.append(rec)
                continue
            rec["fills"] = dump_fills(filled) if filled is not None else []
            if rec["type"] == 1 and not rec["ext"] and ex.order_id_convertor.counter > before_counter:
                # the agent order (or its remainder) rested and got this internal id
                agent_live.append((ex.order_id_convertor.counter, direction, price))
                rec["rested_id"] = ex.order_id_convertor.counter
            seq.append(rec)
        cases.append(dict(init=[[0 if o.direction == "buy" else 1, int(o.price), int(o.volume)] for o in init],
                          orders=seq, dead=dead, book=dump_book(ex.central_orderbook),
                          agent_book=dump_book(ex.internal_orderbook)))
    save("exchange_fuzz.json.gz", cases)


def golden_packed_fixture():
    """The MSFT 2012-06-21 fixture (first 1000 LOBSTER rows, 50 levels) packed by rl4mm_b200.packing, so that the tests
    can replay it without the reference."""
    from rl4mm_b200.packing import pack_lobster

    arrays = {}
    for tie in ("reference", "file"):
        s = pack_lobster(MSG_CSV, BOOK_CSV, 50, max_rows=1000, tie_order=tie)
        arrays[f"msgs_{tie}"] = s.msgs
        arrays.update(step_off=s.step_off, snapshots=s.snapshots, snap_valid=s.snap_valid, ext_ids=s.ext_ids,
                      t0_us=np.int64(s.t0_us), step_us=np.int64(s.step_us))
    np.savez_compressed(GOLDEN / "msft_fixture_packed.npz", **arrays)


# ---------------------------------------------------------------------------------------------------------------------
def golden_episode_summary():
    """G6: the evaluation path -- generate_trajectory + append_to_episode_summary_dict + get_sharpe of the unmodified
    reference (rl4mm/gym/utils.py:100-190, RewardFunctions.py:10-22) on the MSFT fixture, FixedActionAgent and Teradactyl."""
    import contextlib
    import io

    from rl4mm.agents.baseline_agents import FixedActionAgent, Teradactyl
    from rl4mm.features.Features import Inventory, Spread, Portfolio
    from rl4mm.gym.HistoricalOrderbookEnvironment import HistoricalOrderbookEnvironment
    from rl4mm.gym.order_tracking.InfoCalculators import SimpleInfoCalculator
    from rl4mm.rewards.RewardFunctions import PnL

    utils = refshim.import_eval_utils()
    cases = []
    specs = [
        ("fixed_1212", lambda: FixedActionAgent(np.array([1.0, 2.0, 1.0, 2.0])), dict(kind="fixed", action=[1, 2, 1, 2]), 2),
        ("teradactyl", lambda: Teradactyl(max_inventory=300, default_kappa=8.0, default_omega=0.4, max_kappa=12.0,
                                          exponent=1.5, inventory_index=1),
         dict(kind="teradactyl", max_inventory=300, default_kappa=8.0, default_omega=0.4, max_kappa=12.0, exponent=1.5,
              inventory_index=1), 3),
    ]
    for name, mk_agent, agent_desc, n_iter in specs:
        episode_length = timedelta(seconds=1.5)
        feats = [Spread(), Inventory(max_value=100000)]
        db = make_db("S", "reference")
        sim = make_sim(db, 20, preload=True, episode_length=episode_length, warm_up=max(f.window_size for f in feats))
        start_td = timedelta(seconds=36001.0)
        env = HistoricalOrderbookEnvironment(
            features=feats, ticker="MSFT", step_size=timedelta(seconds=0.1), episode_length=episode_length,
            initial_portfolio=Portfolio(inventory=0, cash=10**7), min_date=DAY, max_date=DAY, min_start_timedelta=start_td,
            max_end_timedelta=start_td + episode_length, simulator=sim, per_step_reward_function=PnL(),
            terminal_reward_function=PnL(), n_levels=50, info_calculator=SimpleInfoCalculator(),
        )
        esd = utils.init_episode_summary_dict()
        sharpes = []
        agent = mk_agent()
        for _ in range(n_iter):                # get_episode_summary_dict_NONPARALLEL, utils.py:193-201 (portfolio carries over)
            with contextlib.redirect_stdout(io.StringIO()):
                d = utils.generate_trajectory(agent=agent, env=env)
                esd = utils.append_to_episode_summary_dict(esd, d)
            sharpes.append(float(utils.get_sharpe(esd["equity_curves"][-1])))
        cases.append(dict(name=name, agent=agent_desc, n_iterations=n_iter, start_seconds=36001.0, episode_steps=15,
                          initial_cash=10**7, sharpe=sharpes,
                          esd=json.loads(json.dumps(esd, cls=utils.NumpyEncoder))))
    save("episode_summary.json.gz", cases)


def golden_rolling_sharpe_1e12():
    """RollingSharpe at the reference's DEFAULT cash (initial_cash = 1e12, rl4mm/helpers/main_helper.py:78).  There the window
    holds AUMs of ~1e12 whose step-to-step returns are 1e-10..1e-8, and get_sharpe (RewardFunctions.py:10-22) takes
    ``np.diff(np.log(aum))``: log(1e12) = 27.6 carries an absolute rounding error of up to one ulp = 3.6e-15, i.e. up to 1e-4
    RELATIVE on such a return -- the reference's own reward depends on whose ``log`` it links (numpy's SIMD loop, glibc, ...).
    Every step records, besides the reward of the unmodified reference: the same formula with glibc's scalar log / exp
    (``reward_libm``), and the first-order bound on |delta reward| between two implementations whose log is good to one ulp
    (``bound``) -- the tolerance tests/ hold the CUDA path and the oracle to."""
    import math
    import sys as _sys

    from rl4mm.rewards.RewardFunctions import RollingSharpe

    def hook(env, rec):
        d = done_flag = rec["done"]
        rf = env.terminal_reward_function if d else env.per_step_reward_function
        rec["reward_libm"], rec["bound"] = None, None
        if not isinstance(rf, RollingSharpe) or rf.n_filled < rf.min_window_size:
            return
        aum = rf.aum_array[~np.isnan(rf.aum_array)]
        n = len(aum) - 1
        if n < 2 or np.min(aum) <= 0:
            return
        logs = [math.log(float(a)) for a in aum]
        r = np.array([math.exp(logs[i + 1] - logs[i]) - 1 for i in range(n)])
        sd = float(np.std(r, ddof=1))
        rec["reward_libm"] = float(np.mean(r) / (sd + _sys.float_info.min))
        ulp = float(np.spacing(np.log(np.max(aum))))
        e = 2.0 * ulp                                  # two implementations, each within one ulp of the true log
        if sd > 0:
            S = abs(rec["reward"])
            rec["bound"] = float(2 * e / (n * sd) + S * 2 * e * math.sqrt(n / (n - 1)) / sd)

    rng = np.random.default_rng(77)
    rand4 = rng.uniform(0.0, 10.0, size=(64, 4)).tolist()
    cases = [
        run_env_case("rolling_sharpe_default_cash", rand4, {}, ("RS", 12, 5), ("RS", 8, 3), features=[14, 9, 0, 7], n_episodes=3,
                     episode_seconds=1.0, start_seconds=36001.0, portfolio=(0, 1e12), step_hook=hook),
        run_env_case("rolling_sharpe_default_cash_inventory", rand4[9:], {}, ("RS", 20, 4), ("RS", 20, 4), features=[14, 9, 0, 7],
                     episode_seconds=1.5, start_seconds=36001.0, portfolio=(500, 1e12), step_hook=hook),
    ]
    save("rolling_sharpe_1e12.json.gz", cases)


def golden_episode_starts():
    """Seeded episode starts of the unmodified reference (HOE.py:196,333-351: np.random.choice over the business days, then
    np.random.randint over the step offsets, from numpy's GLOBAL state): for a few np.random.seed values the first four
    ``_get_random_start_time()`` of an env -- one trading day, and a two-week date range."""
    from rl4mm.gym.HistoricalOrderbookEnvironment import HistoricalOrderbookEnvironment

    out = []
    for min_date, max_date, t0, t1, ep in ((DAY, DAY, timedelta(hours=10), timedelta(hours=15, minutes=30), timedelta(minutes=30)),
                                           (datetime(2012, 6, 11), datetime(2012, 6, 22), timedelta(hours=9, minutes=45), timedelta(hours=12), timedelta(seconds=90)),
                                           (DAY, DAY, timedelta(hours=10), timedelta(hours=10, minutes=1), timedelta(minutes=1))):
        db = make_db("S", "reference")
        sim = make_sim(db, 20, preload=True, episode_length=ep, warm_up=timedelta(0))
        env = HistoricalOrderbookEnvironment(ticker="MSFT", step_size=timedelta(seconds=0.1), episode_length=ep, min_date=min_date,
                                             max_date=max_date, min_start_timedelta=t0, max_end_timedelta=t1, simulator=sim, n_levels=50)
        for seed in range(6):
            np.random.seed(seed)
            out.append(dict(seed=seed, min_date=min_date.isoformat(), max_date=max_date.isoformat(), min_start_s=t0.total_seconds(),
                            max_end_s=t1.total_seconds(), episode_s=ep.total_seconds(),
                            starts=[env._get_random_start_time().isoformat() for _ in range(4)]))
    save("episode_starts.json.gz", out)


def golden_generator_merge():
    """Multi-generator merge (rl4mm/simulation/OrderbookSimulator.py:137-148): random 2- and 3-generator step windows through
    the reference's own ``OrderbookSimulator._compress_order_dict`` with the reference's Order dataclasses.  Timestamps are
    drawn from a handful of microseconds, and orders are sometimes duplicated across generators, so that the lexicographic
    deque comparison (equal heads defer to the next elements, ties keep the first generator) is what decides."""
    from collections import deque

    from rl4mm.orderbook.create_order import create_order
    from rl4mm.simulation.OrderbookSimulator import OrderbookSimulator

    rng = np.random.default_rng(20260101)
    kinds = {1: "limit", 2: "cancellation", 3: "deletion", 4: "market"}
    cases = []
    for c in range(200):
        n_gen = int(rng.integers(2, 4))
        pool = []                                             # shared pool => cross-generator duplicates
        for _ in range(int(rng.integers(2, 7))):
            pool.append(dict(us=int(rng.integers(1, 5)), type=int(rng.choice([1, 2, 3, 4])), direction=int(rng.choice([-1, 1])),
                             ext_id=int(rng.integers(1, 4)), size=int(rng.integers(1, 3)) * 100, price=int(rng.integers(1, 3)) * 100))
        gens = []
        for g in range(n_gen):
            k = int(rng.integers(1, 6))
            rows = [dict(pool[int(rng.integers(0, len(pool)))]) if rng.random() < 0.6 else
                    dict(us=int(rng.integers(1, 5)), type=int(rng.choice([1, 2, 3, 4])), direction=int(rng.choice([-1, 1])),
                         ext_id=int(rng.integers(1, 50)), size=int(rng.integers(1, 9)) * 100, price=int(rng.integers(1, 9)) * 100)
                    for _ in range(k)]
            rows.sort(key=lambda r: r["us"])                  # a generator hands its orders out in time order
            gens.append(rows)
        od = {}
        for g, rows in enumerate(gens):
            dq = deque()
            for i, r in enumerate(rows):
                o = create_order(kinds[r["type"]], dict(timestamp=DAY + timedelta(hours=10, microseconds=r["us"]), price=r["price"], volume=r["size"],
                                                        direction="buy" if r["direction"] == 1 else "sell", ticker="MSFT", internal_id=None,
                                                        external_id=r["ext_id"], is_external=True))
                o._src = (g, i)
                dq.append(o)
            od[f"gen_{g}"] = dq
        merged = OrderbookSimulator._compress_order_dict(od)
        cases.append(dict(generators=gens, merged=[list(o._src) for o in merged]))
    save("generator_merge.json.gz", cases)


def main():
    refshim.install()
    golden_packed_fixture()
    import warnings

    warnings.simplefilter("ignore")
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):  # the reference prints on resync / clamping
        g1 = golden_fixture_replay
        g1()
        golden_env_episodes()
        golden_env_random()
        golden_beta_ladders()
        golden_exchange_fuzz()
        golden_episode_summary()
        golden_generator_merge()
        golden_rolling_sharpe_1e12()
        golden_episode_starts()
    for p in sorted(GOLDEN.glob("*.gz")):
        print(p.name, p.stat().st_size)


if __name__ == "__main__":
    main()
