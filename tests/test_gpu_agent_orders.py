"""lobsim_get_agent_orders_dev / LobSim.agent_orders: the agent's resting orders of every env and their queue positions, read
on the device in one launch, against the oracle: the orders from its internal book (dump_agent_orders: price, volume, id, in
ascending id), their level and the orders and volume ahead of them from its L3 central book (dump_book; Exchange.py:196-217).
Every field must match exactly: after env steps and fused rollouts, process_orders, an outer-level resync, hand-built books
and on deep-mode blobs in HBM.  A flat blob reads as empty and stays flat, and the read changes nothing: two handles on the
same program, one of which reads before and after every call, stay identical."""
import ctypes
from datetime import datetime

import numpy as np
import pytest

import adversarial_streams as A
import parity_helpers as H
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu

FIELDS = ("count", "price", "volume", "id", "level", "ahead_orders", "ahead_volume")
ID_MASK = 0x7FFFFFFF


def expected(o, max_orders):
    """The oracle's agent orders and queue positions -> count [2] and the six slot fields [2, max_orders].  ``id`` is the
    oracle's internal id, which also numbers the external orders (OrderIDConvertor.py:12-18); the device numbers the agent's
    orders only, so only the order of the ids is common to both."""
    count = np.zeros(2, np.int32)
    price = np.full((2, max_orders), abi.NO_PRICE, np.int32)
    volume, ident, ahead_n = (np.zeros((2, max_orders), np.int32) for _ in range(3))
    level = np.full((2, max_orders), -1, np.int32)
    ahead_v = np.zeros((2, max_orders), np.int64)
    for side in (0, 1):
        pos, k, last, n, v = {}, -1, None, 0, 0          # agent ref -> (level, orders ahead, volume ahead) in the L3 book
        for p, vol, r in zip(*(o.dump_book(side)[f].tolist() for f in ("price", "volume", "ref"))):
            if p != last:
                k, last, n, v = k + 1, p, 0, 0
            if r & abi.REF_AGENT:
                pos[r] = (k, n, v)
            n, v = n + 1, v + vol
        ag = o.dump_agent_orders(side)
        count[side] = len(ag)
        for i, e in enumerate(ag[:max_orders]):
            price[side, i], volume[side, i], ident[side, i] = e["price"], e["volume"], int(e["ref"]) & ID_MASK
            level[side, i], ahead_n[side, i], ahead_v[side, i] = pos.get(int(e["ref"]), (-1, 0, 0))
    return count, price, volume, ident, level, ahead_n, ahead_v


def read(sim, max_orders=None, queue=True):
    return [t.cpu().numpy() for t in sim.agent_orders(max_orders, queue=queue)]


def device_ids(sim, env, max_orders):
    """The ids of the device's internal book (lobsim_dump_agent_orders, ascending), [2, max_orders], 0-padded."""
    out = np.zeros((2, max_orders), np.int32)
    for side in (0, 1):
        ids = (sim.dump_agent_orders(env, side)["ref"] & ID_MASK).astype(np.int32)[:max_orders]
        out[side, : len(ids)] = ids
    return out


def assert_agent_orders(sim, oracles, what, max_orders=None):
    """agent_orders(max_orders) of every env == the oracle's, ids == the device's own host dump.  The read comes first (the
    dumps would convert flat blobs)."""
    got = read(sim, max_orders)
    A_ = got[1].shape[2]
    assert A_ == (sim.cfg.max_agent_orders if max_orders is None else max_orders)
    for env, o in enumerate(oracles):
        want = list(expected(o, A_))
        want[3] = device_ids(sim, env, A_)
        for name, g, w in zip(FIELDS, got, want):
            assert np.array_equal(g[env], w), (what, env, name, g[env], w)
    return got


def env_kw(**extra):
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(n_levels=10, episode_steps=60, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7, max_levels_per_side=64,
              max_orders_per_side=256)
    kw.update(extra)
    return kw


TERADACTYL = dict(kind=abi.AGENT_TERADACTYL, inventory_index=1, max_inventory=300.0, default_kappa=7.0, default_omega=0.4,
                  max_kappa=12.0, exponent=1.5)


@pytest.mark.parametrize("agent_kind", ["external", "fixed", "teradactyl"])
def test_env_steps_and_rollouts_match_oracle(agent_kind, kernel_family):
    """The agent's ladders after env steps (random actions) or fused FixedAction / Teradactyl rollouts: every field of every
    slot == the oracle after every call, with orders behind others and on several levels seen."""
    import torch

    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=3, n_msgs=60_000, duration_s=200))
    kw = env_kw()
    starts = np.array([200, 500, 900, 1400], np.int32)
    n = len(starts)
    sim = make_sim(abi.default_cfg(n_envs=n, **kw), [s])
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(n)]
    sim.reset(0, starts)
    for o, st in zip(oracles, starts):
        o.reset(int(st))
    ad = abi.action_dim(sim.cfg)
    rng = np.random.default_rng(11)
    if agent_kind == "fixed":
        agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
    elif agent_kind == "teradactyl":
        agent = abi.Agent(**TERADACTYL)
    behind, levels = 0, set()
    for t in range(12):
        if agent_kind == "external":
            a = rng.uniform(0.5, 6.0, size=(n, ad))
            sim.step(torch.tensor(a, device="cuda"))
            for env, o in enumerate(oracles):
                o.step(a[env])
        else:
            sim.rollout(3, agent)
            for o in oracles:
                o.rollout(3, agent)
        got = assert_agent_orders(sim, oracles, (agent_kind, t))
        behind += int(np.count_nonzero(got[5]))
        levels |= set(got[4][got[4] >= 0].tolist())
    assert behind > 0, "some agent orders rest behind others"
    assert len(levels) > 1, levels
    sim.close()


def _gap_price(buy_prices, tick):
    """A buy price strictly between two levels of the side (levels best first)."""
    for hi, lo in zip(buy_prices, buy_prices[1:]):
        if hi - lo > tick:
            return hi - tick
    return buy_prices[-1] - tick


def test_process_orders_fills_and_cancels(kernel_family):
    """Agent limits at the best price (three of them), behind it, at a new price between levels and on the sell side; an
    external market order that eats half of what rests ahead, then one that fills the first agent order in part; agent
    cancels (partial and full).  Compared after every call."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=7, n_msgs=60_000, duration_s=200))
    kw = dict(n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32)
    starts = np.array([300, 800, 1300], np.int32)
    n = len(starts)
    sim = make_sim(abi.default_cfg(n_envs=n, **kw), [s])
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in range(n)]
    sim.reset_book(0, starts)
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    sim.replay(37)
    for o in oracles:
        o.replay(37)
    assert_agent_orders(sim, oracles, "replayed")

    oracle_id = [{} for _ in range(n)]        # device agent id -> the oracle's internal id, per env

    def run(orders, what):
        refs = sim.process_orders(np.array(orders, abi.ORDER_DTYPE))[1]
        for (env, typ, side, px, vol, ext, ref, _), r in zip(orders, refs):
            oid = oracles[env].process_order(typ, side, px, vol, ext, oracle_id[env][ref] if ref and not ext else ref)
            if typ == abi.MSG_LIMIT and not ext:
                assert (r == 0) == (oid == 0), what
                oracle_id[env][int(r)] = oid
        return assert_agent_orders(sim, oracles, what), refs

    orders, ahead_first = [], []
    for env, o in enumerate(oracles):
        buy, sell = o.dump_book(0), o.dump_book(1)
        bb, bs = int(buy["price"][0]), int(sell["price"][0])
        gap = _gap_price(sorted(set(buy["price"].tolist()), reverse=True), 100)
        ahead_first.append(int(buy["volume"][buy["price"] == bb].sum()))
        for side, px, vol in ((0, bb, 37), (0, bb, 12), (0, bb, 9), (0, bb - 200, 5), (0, gap, 8), (1, bs, 11), (1, bs, 4),
                              (1, bs + 1300, 3)):
            orders.append((env, abi.MSG_LIMIT, side, px, vol, 0, 0, 0))
    got, refs = run(orders, "limits")
    assert np.all(got[0][:, 0] == 5) and np.all(got[0][:, 1] == 3)
    assert np.all(got[5][:, 0, 0] > 0) and np.all(got[4][:, 0, 0] == 0)
    assert np.all(got[5][:, 0, 1] == got[5][:, 0, 0] + 1) and np.all(got[6][:, 0, 2] == got[6][:, 0, 0] + 49)
    # external market sells: half of what rests ahead of the first agent order, then the rest of it and 10 of the agent's 37
    half = [(env, abi.MSG_MARKET, 1, 0, max(1, v // 2), 1, 0, 0) for env, v in enumerate(ahead_first)]
    got2, _ = run(half, "market half")
    assert np.all(got2[6][:, 0, 0] < got[6][:, 0, 0])
    rest = [(env, abi.MSG_MARKET, 1, 0, int(got2[6][env, 0, 0]) + 10, 1, 0, 0) for env in range(n)]
    got3, _ = run(rest, "market into the agent")
    assert np.all(got3[2][:, 0, 0] == 27) and np.all(got3[5][:, 0, 0] == 0) and np.all(got3[6][:, 0, 1] == 27)
    # agent cancels: 5 of the second order at the best price, the whole order behind it, the first sell order
    cancels = []
    for env in range(n):
        ids = refs[env * 8: env * 8 + 8]
        p = got3[1][env, 0]
        cancels += [(env, abi.MSG_CANCEL, 0, int(p[1]), 5, 0, int(ids[1]), 0), (env, abi.MSG_DELETE, 0, int(p[3]), 0, 0, int(ids[3]), 0),
                    (env, abi.MSG_DELETE, 1, int(got3[1][env, 1, 0]), 0, 0, int(ids[5]), 0)]
    got4, _ = run(cancels, "cancels")
    assert np.all(got4[0][:, 0] == 4) and np.all(got4[0][:, 1] == 2) and np.all(got4[2][:, 0, 1] == 7)
    sim.close()


def test_resync_requeues_behind_the_aggregate(kernel_family):
    """testOrderbookSimulator.py:77-108: agent orders at prices that update_outer_levels overwrites are cancelled and re-queued
    behind the snapshot aggregate, so the aggregate is ahead of them."""
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim
    from rl4mm_b200.simulation import DeviceDatabase

    db = DeviceDatabase()
    db.add_stream("MSFT", datetime(2012, 6, 21), H.load_fixture_stream("reference"))
    stream = db.streams[0]
    start = db.step_of(0, datetime(2012, 6, 21, 10, 0, 0))
    kw = dict(n_levels=50, outer_levels=48, resync=1)
    n = 2
    sim = LobSim(abi.default_cfg(n_envs=n, **kw), 0)
    sim.load_stream(0, stream)
    sim.reset_book(0, np.full(n, start, np.int32))
    oracles = [Oracle(abi.default_cfg(**kw), stream) for _ in range(n)]
    for o in oracles:
        o.reset_book(start)
    worst_buy, worst_sell = int(oracles[0].dump_book(0)["price"][-1]), int(oracles[0].dump_book(1)["price"][-1])
    orders = [(env, abi.MSG_LIMIT, side, px, vol, 0, 0, 0) for env in range(n) for side, px, vol in ((0, worst_buy - 100, 100),
                                                                                                      (1, worst_sell, 200))]
    sim.process_orders(np.array(orders, abi.ORDER_DTYPE))
    for env, typ, side, px, vol, ext, ref, _ in orders:
        oracles[env].process_order(typ, side, px, vol, ext, ref)
    before = assert_agent_orders(sim, oracles, "placed")
    assert np.all(before[5][:, 0, 0] == 0)                          # alone at a new price
    sim.forward_step(stream.steps_per_second)
    for o in oracles:
        o.forward_step(stream.steps_per_second)
    got = assert_agent_orders(sim, oracles, "resynced")
    assert np.all(got[1][:, 0, 0] == worst_buy - 100) and np.all(got[2][:, 0, 0] == 100)
    assert np.all(got[5][:, 0, 0] == 1) and np.all(got[6][:, 0, 0] == 200), (got[5][:, 0], got[6][:, 0])
    sim.close()


def test_set_book_hand_built(kernel_family):
    """Agent, external and aggregate orders interleaved in one level, five 1e9-sized orders ahead of an agent order (volume
    ahead beyond 2^32), 40 agent orders on 40 sell levels whose ids fall as the price worsens (more than one group of 32),
    and a read with max_orders below the count: the count stays the full count and the first ids are written."""
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    p, G = 1_000_000, 10**9
    ag = abi.REF_AGENT
    # inside a level the agent ids rise along the FIFO (time priority), as they would in a real book
    buy = [(p, G, 0), (p, G, 7), (p, G, 8), (p, 5, ag | 3), (p, 2 * G, 9), (p, 7, ag | 10), (p, 3, ag | 50),
           (p - 100, 4, ag | 2), (p - 300, 2, 10), (p - 300, 3, ag | 5), (p - 300, 1, 11), (p - 400, 6, 12)]
    sell = []
    for k in range(40):
        sell += [(p + 100 * (k + 1), k + 1, 100 + k), (p + 100 * (k + 1), 2, ag | (99 - k))]
        if k % 3 == 0:
            sell.append((p + 100 * (k + 1), 9, 200 + k))
    buy = np.array([e + (0,) for e in buy], abi.BOOK_ENTRY_DTYPE)
    sell = np.array([e + (0,) for e in sell], abi.BOOK_ENTRY_DTYPE)
    kw = dict(n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=64)
    sim = LobSim(abi.default_cfg(n_envs=3, **kw), 0)
    sim.set_book(1, buy, sell)
    sim.set_book(2, sell[:0], sell)
    oracles = [Oracle(abi.default_cfg(**kw)) for _ in range(3)]
    oracles[1].set_book(buy, sell)
    oracles[2].set_book(sell[:0], sell)
    got = assert_agent_orders(sim, oracles, "set_book")
    assert list(got[0][1]) == [5, 40] and list(got[0][2]) == [0, 40] and list(got[0][0]) == [0, 0]
    assert list(got[3][1, 0, :5]) == [2, 3, 5, 10, 50] and list(got[3][1, 1, :40]) == list(range(60, 100))
    assert list(got[5][1, 0, :5]) == [0, 3, 1, 5, 6] and got[6][1, 0, 1] == 3 * G and got[6][1, 0, 3] == 5 * G + 5
    assert list(got[4][1, 0, :5]) == [1, 0, 2, 0, 0]
    assert list(got[4][1, 1, :40]) == list(range(39, -1, -1))
    for m in (1, 8, 33):
        small = assert_agent_orders(sim, oracles, ("max_orders", m), max_orders=m)
        assert list(small[0][1]) == [5, 40]
        for g, w in zip(small[1:], got[1:]):
            assert np.array_equal(g, w[:, :, :m]), m
    sim.close()


@pytest.mark.fast_only        # deep-book capacities always run the general kernel on the blobs in HBM
def test_deep_books_in_hbm():
    """256 levels x 16 384 orders per side (deep-mode blobs in HBM, queues of ~80 orders): Teradactyl and FixedAction
    rollouts, then every field == the oracle, with queues ahead longer than one 32-entry round."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    sc = synthetic.SynthConfig(seed=11, n_msgs=300_000, duration_s=600, n_levels=50, mid0=2_000_000, p_limit=0.40, p_cancel=0.15,
                               p_delete=0.37, p_exec=0.08, geom_p=0.10, init_levels=70, mean_queue=80, target_orders=6000,
                               max_offset_ticks=80)
    s = synthetic.generate(sc)
    kw = env_kw(n_levels=50, outer_levels=20, max_levels_per_side=256, max_orders_per_side=16384)
    starts = np.array([100, 1500, 3000], np.int32)
    sim = make_sim(abi.default_cfg(n_envs=len(starts), max_agent_orders=64, **kw), [s])
    assert sim.kernel_path == "deep"
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(len(starts))]
    sim.reset(0, starts)
    for o, st in zip(oracles, starts):
        o.reset(int(st))
    far = 0
    for agent in (abi.Agent(**TERADACTYL), abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))):
        for _ in range(3):
            sim.rollout(4, agent)
            for o in oracles:
                o.rollout(4, agent)
            got = assert_agent_orders(sim, oracles, "deep")
            far = max(far, int(got[5].max()))
    assert far > 32, far
    sim.close()


def test_flat_blobs_read_empty_and_stay_flat(kernel_family):
    """Thin books replayed by the straight-line kernel stay in the flat form between launches.  The read returns count 0 and
    empty slots, and leaves the blobs flat."""
    from rl4mm_b200.device import LobSim

    shape = "thin"
    s = A.build(shape, A.SHAPES[shape]["seeds"][0])
    starts = [10 * t for t in A.STARTS]
    cfg = A.cfg_for(shape, n_envs=len(starts), resync=0, outer_levels=2)
    sim = LobSim(cfg, 0)
    sim.load_stream(0, s)
    sim.reset_book(0, np.array(starts, np.int32))
    flat_reads, done = 0, 0
    while done < min(s.n_grid_steps, 200):
        sim.replay(7)
        done += 7
        flat_before = sim.state()["reserved"] & 1
        got = read(sim)
        assert np.array_equal(sim.state()["reserved"] & 1, flat_before), done
        flat_reads += int(flat_before.sum())
        assert not got[0].any() and np.all(got[1] == abi.NO_PRICE) and np.all(got[4] == -1), done
        assert not got[2].any() and not got[3].any() and not got[5].any() and not got[6].any(), done
    if kernel_family == "fast":
        assert flat_reads > 0, "flat blobs were read"
    sim.close()


def test_read_has_no_side_effects(kernel_family):
    """Handles A and B run the same program (replay, env steps, rollouts, replay again); A reads the agent orders before and
    after every call, B never does.  State (book form bit included), errors, obs, rewards and the final books are identical,
    and every read is exactly one launch."""
    import torch

    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=5, n_msgs=60_000, duration_s=200))
    kw = env_kw(episode_steps=40)
    n = 6
    a, b = make_sim(abi.default_cfg(n_envs=n, **kw), [s]), make_sim(abi.default_cfg(n_envs=n, **kw), [s])
    starts = np.array([100, 300, 500, 700, 900, 1100], np.int32)
    rng = np.random.default_rng(2)
    acts = [torch.tensor(rng.uniform(0.5, 6.0, size=(n, abi.action_dim(a.cfg))), device="cuda") for _ in range(4)]
    agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
    program = [lambda h: h.reset_book(0, starts), lambda h: h.replay(7), lambda h: h.replay(23), lambda h: h.reset(0, starts + 100)]
    program += [lambda h, x=x: h.step(x) for x in acts]
    program += [lambda h: h.rollout(5, agent), lambda h: h.rollout(3, abi.Agent(**TERADACTYL)), lambda h: h.reset_book(0, starts + 50),
                lambda h: h.replay(31), lambda h: h.replay(3)]
    flat_reads, seen = 0, 0
    for i, call in enumerate(program):
        for kwargs in (dict(), dict(max_orders=1, queue=False)):
            c = a.launch_count
            a.agent_orders(**kwargs)
            assert a.launch_count == c + 1, (i, kwargs)
        flat_reads += int(np.sum(a.state()["reserved"] & 1))
        ra, rb = call(a), call(b)
        if isinstance(ra, tuple):
            for x, y in zip(ra, rb):
                assert torch.equal(x, y), i
        elif isinstance(ra, torch.Tensor):
            assert torch.equal(ra, rb), i
        c = a.launch_count
        seen += int(a.agent_orders()[0].sum())
        assert a.launch_count == c + 1, i
        assert torch.equal(a.state_dev(), b.state_dev()), i
        assert np.array_equal(a.errors(), b.errors()), i
    assert seen > 0
    if kernel_family == "fast":
        assert flat_reads > 0, "some reads found flat blobs pending"
    for env in range(n):
        for side in (0, 1):
            assert np.array_equal(a.dump_book(env, side), b.dump_book(env, side)), (env, side)
            assert np.array_equal(a.dump_agent_orders(env, side), b.dump_agent_orders(env, side)), (env, side)
    a.close()
    b.close()


def test_cuda_graph_capture(kernel_family):
    """step_torch + agent_orders(out=...) captured once in a CUDA graph and replayed k times == an eager twin."""
    from datetime import timedelta

    import torch

    from rl4mm_b200 import synthetic
    from rl4mm_b200.features import Inventory, Portfolio, Spread
    from rl4mm_b200.gym import HistoricalOrderbookEnvironment
    from rl4mm_b200.rewards import PnL
    from rl4mm_b200.simulation import DeviceDatabase

    s = synthetic.generate(synthetic.spy_day(seed=21, n_msgs=80_000, duration_s=300))
    day = datetime(2019, 1, 2)
    db = DeviceDatabase()
    db.add_stream("SPY", day, s)

    def make_env():
        return HistoricalOrderbookEnvironment(
            features=[Spread(), Inventory()], ticker="SPY", episode_length=timedelta(seconds=20), min_date=day, max_date=day,
            min_start_timedelta=timedelta(hours=9, minutes=30, seconds=5), max_end_timedelta=timedelta(hours=9, minutes=34),
            initial_portfolio=Portfolio(inventory=0, cash=10**7), per_step_reward_function=PnL(), terminal_reward_function=PnL(),
            n_levels=10, database=db, n_envs=40, max_levels_per_side=64, max_orders_per_side=256, seed=9)

    g_env, e_env = make_env(), make_env()
    g_env.reset()
    e_env.reset()
    assert np.array_equal(g_env.episode_start_steps, e_env.episode_start_steps)
    rng = np.random.default_rng(4)
    action = torch.tensor(rng.uniform(0.5, 6.0, size=(40, 4)), device="cuda")
    A_ = 24
    sl = (40, 2, A_)
    out = (torch.empty((40, 2), dtype=torch.int32, device="cuda"),) + tuple(torch.empty(sl, dtype=torch.int32, device="cuda")
                                                                           for _ in range(5)) \
        + (torch.empty(sl, dtype=torch.int64, device="cuda"),)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):              # warm-up step outside the graph (eager twin: the same step)
        g_env.step_torch(action)
        g_env.agent_orders(A_, out=out)
    torch.cuda.current_stream().wait_stream(side)
    e_env.step_torch(action)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obs_g, rew_g, _ = g_env.step_torch(action)
        g_env.agent_orders(A_, out=out)
    for k in range(6):
        graph.replay()
        obs_e, rew_e, _ = e_env.step_torch(action)
        want = e_env.agent_orders(A_)
        torch.cuda.synchronize()
        assert torch.equal(obs_g, obs_e) and torch.equal(rew_g, rew_e), k
        for name, g, w in zip(FIELDS, out, want):
            assert torch.equal(g, w), (k, name)
    assert bool((out[0] > 0).any()) and bool((out[5] > 0).any()), "the agent's resting orders are read in the graph"


def test_arguments_and_fresh_handle(kernel_family):
    """A fresh handle reads count 0 and empty slots; max_orders outside [1, max_agent_orders] and NULL required pointers are
    LOBSIM_E_INVALID (LobsimError in the façade) without a launch; the queue outputs may be NULL; out= is checked."""
    import torch

    from rl4mm_b200._lib import LobsimError, lib
    from rl4mm_b200.device import LobSim

    sim = LobSim(abi.default_cfg(n_envs=5, n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32), 0)
    got = read(sim)
    assert [g.shape for g in got] == [(5, 2)] + [(5, 2, 32)] * 6
    assert [g.dtype for g in got] == [np.int32] * 6 + [np.int64]
    assert not got[0].any() and np.all(got[1] == abi.NO_PRICE) and np.all(got[4] == -1)
    assert not got[2].any() and not got[3].any() and not got[5].any() and not got[6].any()
    assert len(sim.agent_orders(3, queue=False)) == 4
    for bad in (0, -1, 33):
        with pytest.raises(LobsimError):
            sim.agent_orders(bad)
    t = sim.agent_orders(3)
    ptr = [ctypes.c_void_p(x.data_ptr()) for x in t]
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = lib()
    assert L.lobsim_get_agent_orders_dev(sim._h, 3, *ptr[:4], None, None, None, st) == abi.OK
    assert L.lobsim_get_agent_orders_dev(sim._h, 3, *ptr, st) == abi.OK
    for m, null in ((0, None), (33, None), (3, 0), (3, 1), (3, 2), (3, 3)):
        args = list(ptr)
        if null is not None:
            args[null] = None
        c = sim.launch_count
        assert L.lobsim_get_agent_orders_dev(sim._h, m, *args, st) == abi.E_INVALID, (m, null)
        assert sim.launch_count == c
    assert L.lobsim_get_agent_orders_dev(None, 3, *ptr, st) == abi.E_INVALID
    with pytest.raises(ValueError):
        sim.agent_orders(3, out=t[:4])                                        # queue=True wants seven tensors
    with pytest.raises(ValueError):
        sim.agent_orders(3, out=t[:6] + (t[6].to(torch.int32),))              # dtype
    with pytest.raises(ValueError):
        sim.agent_orders(2, out=t)                                            # shape
    with pytest.raises(ValueError):
        sim.agent_orders(3, out=(t[0].cpu(),) + t[1:])                        # device
    assert sim.agent_orders(3, out=t) is not None
    sim.close()
