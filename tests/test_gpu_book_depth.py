"""lobsim_get_depth_dev / LobSim.book_depth: the L2 depth of every book, read on the device in one launch, against the L2
projection of the oracle's L3 book (rl4mm/extras/orderbook_comparison.py:6-19): group by price, best first, absent levels
(NO_PRICE, 0).  Price, volume, queue length and the agent's volume must match exactly, on flat blobs (read between replay
launches, never converted), sorted blobs, hybrid-replayed blobs, deep-mode blobs in HBM and books of dead envs.  The read must
change nothing: two handles on the same program, one of which reads before and after every call, stay identical."""
import ctypes

import numpy as np
import pytest

import adversarial_streams as A
import parity_helpers as H
import random_cases as R
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu

FIELDS = ("price", "volume", "orders", "agent_volume")


def l2_of(sides, depth):
    """[buy entries, sell entries] in the dump_book format (best level first) -> price, volume, orders, agent_volume [2, depth]."""
    out = (np.full((2, depth), abi.NO_PRICE, np.int32), np.zeros((2, depth), np.int64), np.zeros((2, depth), np.int32),
           np.zeros((2, depth), np.int64))
    for side, e in enumerate(sides):
        k, last = -1, None
        for p, v, r in zip(e["price"].tolist(), e["volume"].tolist(), e["ref"].tolist()):
            if p != last:
                k, last = k + 1, p
            if k >= depth:
                break
            out[0][side, k] = p
            out[1][side, k] += v
            out[2][side, k] += 1
            if r & abi.REF_AGENT:
                out[3][side, k] += v
    return out


def oracle_l2(o, depth):
    return l2_of([o.dump_book(0), o.dump_book(1)], depth)


def read(sim, depth):
    return [t.cpu().numpy() for t in sim.book_depth(depth, orders=True, agent=True)]


def assert_depth(sim, oracles, depth, what, dead_as_is=False, cfg=None):
    """book_depth(depth) of every env == the oracle's L2 book.  The read comes first (flat blobs are read as they are: the L3
    dumps below would convert them).  Envs whose device book hit a capacity are left out; with ``dead_as_is`` the book of an
    env the reference would have raised on (EmptyOrderbookError) is compared with its own device L3 dump instead."""
    got = read(sim, depth)
    st = sim.state()
    for env, o in enumerate(oracles):
        if cfg is not None and H.capacity_excluded(st["err"][env], o, cfg, (what, env)):
            continue
        if dead_as_is and int(o.state()["err"]) & abi.ERR_EMPTY_BOOK:
            want = l2_of([sim.dump_book(env, 0), sim.dump_book(env, 1)], depth)
        else:
            want = oracle_l2(o, depth)
        for name, g, w in zip(FIELDS, got, want):
            assert np.array_equal(g[env], w), (what, env, depth, name, g[env], w)
    return st


@pytest.mark.replay_path
@pytest.mark.parametrize("seed", [2, 13, 15, 19, 20, 21])
def test_depth_after_ragged_replays_matches_oracle(seed, kernel_family):
    """Random replay cases (thin books, books around the flat pool capacity, deep books): depth 1, n_levels and
    max_levels_per_side after every launch of a ragged replay."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    c = R.random_replay_case(seed)
    s = synthetic.generate(c["synth"])
    n = c["n_envs"]
    okw = {k: v for k, v in c["cfg_kw"].items() if not k.startswith("max_")}
    cfg = abi.default_cfg(n_envs=n, **c["cfg_kw"])
    sim = make_sim(cfg, [s])
    oracles = [Oracle(abi.default_cfg(n_envs=1, **okw), s) for _ in range(n)]
    sim.reset_book(0, c["starts"])
    for o, st in zip(oracles, c["starts"]):
        o.reset_book(int(st))
    depths = (1, s.n_levels, cfg.max_levels_per_side)
    flat_seen = False
    for chunk in c["chunks"]:
        sim.replay(chunk)
        for o in oracles:
            o.replay(chunk)
        for depth in depths:
            st = assert_depth(sim, oracles, depth, (seed, chunk), cfg=cfg)
            flat_seen |= bool(np.any(st["reserved"] & 1))
    if kernel_family == "fast" and sim.kernel_path == "fast" and c["synth"].target_orders <= 30:
        assert flat_seen, "thin books are read in the flat form"
    sim.close()


STREAMS = [(shape, seed) for shape, sh in A.SHAPES.items() for seed in sh["seeds"]]


@pytest.mark.replay_path
@pytest.mark.parametrize("shape,seed", STREAMS)
def test_depth_on_adversarial_streams(shape, seed, kernel_family):
    """Sides emptied by sweeps, EmptyOrderbookError in the middle of a second (dead books are read as they are), full flat
    pools, and the capacities without a compiled layout (96/384/32): depth after every ragged replay launch."""
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    s = A.build(shape, seed)
    starts = [10 * t for t in A.STARTS]
    cfg = A.cfg_for(shape, n_envs=len(starts), resync=0, outer_levels=2)
    sim = LobSim(cfg, 0)
    sim.load_stream(0, s)
    sim.reset_book(0, np.array(starts, np.int32))
    oracles = [Oracle(A.cfg_for(shape, resync=0, outer_levels=2), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    done, k, flat_reads = 0, 0, 0
    while done < s.n_grid_steps:
        chunk = (1, 3, 7, 10, 23, 57)[k % 6]
        k += 1
        sim.replay(chunk)
        for o in oracles:
            o.replay(chunk)
        done += chunk
        st = assert_depth(sim, oracles, s.n_levels, (shape, seed, done), dead_as_is=True)
        flat_reads += int(np.sum(st["reserved"] & 1))
    st = assert_depth(sim, oracles, cfg.max_levels_per_side, (shape, seed, "end"), dead_as_is=True)
    assert np.any(st["err"] & abi.ERR_EMPTY_BOOK), "the stream kills at least one of its books"
    if shape == "thin" and kernel_family in ("fast", "hybrid"):
        assert flat_reads > 0, "flat blobs were read"
    sim.close()


@pytest.mark.parametrize("agent_kind", ["external", "fixed"])
def test_agent_volume_and_queue_lengths_match_oracle(agent_kind, kernel_family):
    """The agent's ladders resting in the books (env steps or a FixedAction rollout), then lobsim_process_orders with agent
    limits at existing and at new prices: orders and agent_volume per level == the oracle's."""
    import torch

    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=3, n_msgs=60_000, duration_s=200))
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(n_levels=10, episode_steps=60, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7, max_levels_per_side=64, max_orders_per_side=256)
    starts = np.array([200, 500, 900, 1400], np.int32)
    n = len(starts)
    sim = make_sim(abi.default_cfg(n_envs=n, **kw), [s])
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(n)]
    sim.reset(0, starts)
    for o, st in zip(oracles, starts):
        o.reset(int(st))
    ad = abi.action_dim(sim.cfg)
    rng = np.random.default_rng(11)
    agent_seen = 0
    for t in range(12):
        if agent_kind == "external":
            a = rng.uniform(0.5, 6.0, size=(n, ad))
            sim.step(torch.tensor(a, device="cuda"))
            for env, o in enumerate(oracles):
                o.step(a[env])
        else:
            agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
            sim.rollout(3, agent)
            for o in oracles:
                o.rollout(3, agent)
        got = read(sim, 10)
        assert_depth(sim, oracles, 10, (agent_kind, t))
        agent_seen += int(np.count_nonzero(got[3]))
    assert agent_seen > 0, "the agent's orders rest at the central levels"
    # agent limits at the best price, two ticks behind it and at a price between the levels of the buy side
    st = sim.state()
    orders, orc = [], []
    for env in range(n):
        bb, bs = int(st["best_buy"][env]), int(st["best_sell"][env])
        for side, px, vol in ((0, bb, 37), (0, bb - 200, 5), (1, bs, 11), (1, bs + 1300, 3), (0, bb - 4100, 8)):
            orders.append((env, abi.MSG_LIMIT, side, px, vol, 0, 0, 0))
            orc.append((env, side, px, vol))
    sim.process_orders(np.array(orders, abi.ORDER_DTYPE))
    for env, side, px, vol in orc:
        oracles[env].process_order(abi.MSG_LIMIT, side, px, vol, 0, 0)
    for depth in (1, 10, 64):
        assert_depth(sim, oracles, depth, (agent_kind, "process_orders"))
    sim.close()


def _three_giants_stream(p):
    """One second, 10 levels: a snapshot with a 1e9 aggregate at buy price p, then two more buy limits of 1e9 at p."""
    snaps = np.zeros((2, 2, 10, 2), np.int32)
    snaps[..., 0] = abi.NO_PRICE
    snaps[:, 0, 0], snaps[:, 0, 1], snaps[:, 1, 0] = (p, 10**9), (p - 100, 5), (p + 100, 7)
    msgs = np.zeros(2, abi.MSG_DTYPE)
    msgs["price"], msgs["volume"], msgs["ref"] = p, 10**9, [1, 2]
    msgs["meta"] = abi.meta(abi.MSG_LIMIT, abi.BUY)
    step_off = np.full(11, 2, np.uint32)
    step_off[0] = 0
    from rl4mm_b200.packing import PackedStream

    s = PackedStream(msgs, step_off, snaps, np.ones(2, np.uint8), 0, 100_000, 10)
    s.validate()
    return s


def test_volume_is_int64(kernel_family):
    """Three orders of 1e9 at one price: 3e9 exactly, from set_book (sorted form) and after a replay launch (flat form in the
    fast family)."""
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    p = 1_000_000
    s = _three_giants_stream(p)
    kw = dict(n_levels=10, resync=0, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32)
    sim = LobSim(abi.default_cfg(n_envs=2, **kw), 0)
    sim.load_stream(0, s)
    sim.reset_book(0, 0)
    sim.replay(10)
    o = Oracle(abi.default_cfg(**kw), s)
    o.reset_book(0)
    o.replay(10)
    price, volume, orders, agent = read(sim, 4)
    if kernel_family == "fast":
        assert np.all(sim.state()["reserved"] & 1), "the replay left the books flat"
    want = oracle_l2(o, 4)
    for env in range(2):
        assert price[env, 0, 0] == p and volume[env, 0, 0] == 3 * 10**9 and orders[env, 0, 0] == 3
        for name, g, w in zip(FIELDS, (price, volume, orders, agent), want):
            assert np.array_equal(g[env], w), (env, name)
    buy = np.array([(p, 10**9, 0, 0), (p, 10**9, 7, 0), (p, 10**9, abi.REF_AGENT | 1, 0), (p - 300, 1, 8, 0)], abi.BOOK_ENTRY_DTYPE)
    sell = np.array([(p + 100, 2_000_000_000, 9, 0), (p + 100, 2_000_000_000, 10, 0)], abi.BOOK_ENTRY_DTYPE)
    sim.set_book(1, buy, sell)
    price, volume, orders, agent = read(sim, 2)
    assert not sim.state()["reserved"][1] & 1
    assert list(price[1, 0]) == [p, p - 300] and list(volume[1, 0]) == [3 * 10**9, 1] and list(orders[1, 0]) == [3, 1]
    assert list(agent[1, 0]) == [10**9, 0]
    assert list(price[1, 1]) == [p + 100, abi.NO_PRICE] and list(volume[1, 1]) == [4 * 10**9, 0] and list(orders[1, 1]) == [2, 0]
    sim.close()


@pytest.mark.fast_only        # deep-book capacities always run the general kernel on the blobs in HBM
def test_deep_books_in_hbm():
    """256 levels x 16 384 orders per side (deep-book mode, blobs in HBM, queues of ~80 orders): depth 256 == the oracle."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    sc = synthetic.SynthConfig(seed=11, n_msgs=300_000, duration_s=600, n_levels=50, mid0=2_000_000, p_limit=0.40, p_cancel=0.15,
                               p_delete=0.37, p_exec=0.08, geom_p=0.10, init_levels=70, mean_queue=80, target_orders=6000,
                               max_offset_ticks=80)
    s = synthetic.generate(sc)
    kw = dict(n_levels=50, outer_levels=20)
    starts = [0, 500, 1500]
    sim = make_sim(abi.default_cfg(n_envs=len(starts), max_levels_per_side=256, max_orders_per_side=16384, max_agent_orders=64, **kw), [s])
    assert sim.kernel_path == "deep"
    sim.reset_book(0, np.array(starts, np.int32))
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(st)
    for chunk in (1, 99, 1900):
        sim.replay(chunk)
        for o in oracles:
            o.replay(chunk)
        assert_depth(sim, oracles, 256, ("deep", chunk))
    orders = read(sim, 256)[2]
    assert orders.max() > 100 and orders.sum(axis=2).max() > 1600, (orders.max(), orders.sum(axis=2).max())
    sim.close()


def test_read_has_no_side_effects(kernel_family):
    """Handles A and B run the same program (replay, env steps, rollout, replay again); A reads depth before and after every
    call, B never does.  State (book form bit included), errors, obs, rewards and the final books are identical, and every
    read is exactly one launch -- also while flat blobs are pending, so no conversion ran."""
    import torch

    from rl4mm_b200 import synthetic
    from test_gpu_parity import make_sim

    s = synthetic.generate(synthetic.spy_day(seed=5, n_msgs=60_000, duration_s=200))
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_BOOK_IMBALANCE, 0, 100_000, -1, 1)]
    kw = dict(n_levels=10, episode_steps=40, warmup_steps=10, features=feats, initial_cash=1e7, max_levels_per_side=64,
              max_orders_per_side=256)
    n = 6
    a, b = make_sim(abi.default_cfg(n_envs=n, **kw), [s]), make_sim(abi.default_cfg(n_envs=n, **kw), [s])
    starts = np.array([100, 300, 500, 700, 900, 1100], np.int32)
    rng = np.random.default_rng(2)
    acts = [torch.tensor(rng.uniform(0.5, 6.0, size=(n, abi.action_dim(a.cfg))), device="cuda") for _ in range(4)]
    agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
    program = [lambda h: h.reset_book(0, starts), lambda h: h.replay(7), lambda h: h.replay(23), lambda h: h.reset(0, starts + 100)]
    program += [lambda h, x=x: h.step(x) for x in acts]
    program += [lambda h: h.rollout(5, agent), lambda h: h.reset_book(0, starts + 50), lambda h: h.replay(31), lambda h: h.replay(3)]
    flat_reads = 0
    for i, call in enumerate(program):
        for depth in (1, 10):
            c = a.launch_count
            a.book_depth(depth, orders=depth == 10, agent=depth == 10)
            assert a.launch_count == c + 1, (i, depth)
        flat_reads += int(np.sum(a.state()["reserved"] & 1))
        ra, rb = call(a), call(b)
        if isinstance(ra, tuple):
            for x, y in zip(ra, rb):
                assert torch.equal(x, y), i
        elif isinstance(ra, torch.Tensor):
            assert torch.equal(ra, rb), i
        c = a.launch_count
        a.book_depth(10, orders=True, agent=True)
        assert a.launch_count == c + 1, i
        assert torch.equal(a.state_dev(), b.state_dev()), i
        assert np.array_equal(a.errors(), b.errors()), i
    if kernel_family == "fast":
        assert flat_reads > 0, "some reads found flat blobs pending"
    for env in range(n):
        for side in (0, 1):
            assert np.array_equal(a.dump_book(env, side), b.dump_book(env, side)), (env, side)
            assert np.array_equal(a.dump_agent_orders(env, side), b.dump_agent_orders(env, side)), (env, side)
    a.close()
    b.close()


def test_batched_snapshot_agreement(kernel_family):
    """testOrderbookSimulator.py:46-75 for N replicas at once: book_depth(50) of every env equals the LOBSTER snapshot at t0,
    +1 s and +2 s, with the exclusions of test_agreement_with_lobster (levels the simulated book lacks; buy level 45 at +2 s)."""
    from datetime import datetime

    from rl4mm_b200.device import LobSim
    from rl4mm_b200.simulation import DeviceDatabase, OrderbookSimulator

    db = DeviceDatabase()
    db.add_stream("MSFT", datetime(2012, 6, 21), H.load_fixture_stream("reference"))
    stream = db.streams[0]
    start = db.step_of(0, datetime(2012, 6, 21, 10, 0, 0))
    n = 64
    sim = LobSim(abi.default_cfg(n_envs=n, n_levels=50, outer_levels=48, fill_log_capacity=4096), 0)
    sim.load_stream(0, stream)
    sim.reset_book(0, np.full(n, start, np.int32))
    for sec in (1, 2, 3):
        if sec > 1:
            sim.forward_step(stream.steps_per_second)
        price, volume = (t.cpu().numpy() for t in sim.book_depth(50))
        snap = stream.snapshots[sec]
        for env in range(n):
            keep = np.ones((2, 50), bool) if sec == 1 else price[env] != abi.NO_PRICE
            if sec == 3:
                keep[0, 45] = False
            assert keep.sum() > 90
            assert np.array_equal(price[env][keep], snap[..., 0][keep]), (sec, env)
            assert np.array_equal(volume[env][keep], snap[..., 1][keep].astype(np.int64)), (sec, env)
    sim.close()
    one = OrderbookSimulator("MSFT", None, None, 50, db, preload_orders=False, outer_levels=48)
    one.reset_episode(datetime(2012, 6, 21, 10, 0, 0))
    price, volume = one.book_depth(50)
    assert price.shape == (1, 2, 50) and volume.dtype.itemsize == 8             # batched, not squeezed
    assert np.array_equal(price[0].cpu().numpy(), stream.snapshots[1][..., 0])
    assert np.array_equal(volume[0].cpu().numpy(), stream.snapshots[1][..., 1])


def test_cuda_graph_capture(kernel_family):
    """step_torch + book_depth(out=...) captured once in a CUDA graph and replayed k times == an eager twin."""
    from datetime import datetime, timedelta

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
    depth = 8
    out = (torch.empty((40, 2, depth), dtype=torch.int32, device="cuda"), torch.empty((40, 2, depth), dtype=torch.int64, device="cuda"),
           torch.empty((40, 2, depth), dtype=torch.int32, device="cuda"), torch.empty((40, 2, depth), dtype=torch.int64, device="cuda"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):              # warm-up step outside the graph (eager twin: the same step)
        g_env.step_torch(action)
        g_env.book_depth(depth, orders=True, agent=True, out=out)
    torch.cuda.current_stream().wait_stream(side)
    e_env.step_torch(action)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obs_g, rew_g, _ = g_env.step_torch(action)
        g_env.book_depth(depth, orders=True, agent=True, out=out)
    for k in range(6):
        graph.replay()
        obs_e, rew_e, _ = e_env.step_torch(action)
        want = e_env.book_depth(depth, orders=True, agent=True)
        torch.cuda.synchronize()
        assert torch.equal(obs_g, obs_e) and torch.equal(rew_g, rew_e), k
        for name, g, w in zip(FIELDS, out, want):
            assert torch.equal(g, w), (k, name)
    assert bool((out[3] > 0).any()), "the agent's ladders are part of the depth read in the graph"


def test_arguments_and_fresh_handle(kernel_family):
    """A fresh handle reads all NO_PRICE / 0; depth 0, depth above max_levels_per_side and NULL required pointers are
    LOBSIM_E_INVALID (LobsimError in the façade); the optional outputs may be NULL."""
    import torch

    from rl4mm_b200._lib import LobsimError, lib
    from rl4mm_b200.device import LobSim

    sim = LobSim(abi.default_cfg(n_envs=5, n_levels=10, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32), 0)
    price, volume, orders, agent = read(sim, 64)
    assert price.shape == (5, 2, 64) and np.all(price == abi.NO_PRICE)
    assert not volume.any() and not orders.any() and not agent.any()
    p, v = sim.book_depth(3)
    assert p.dtype == torch.int32 and v.dtype == torch.int64 and p.shape == v.shape == (5, 2, 3)
    for bad in (0, -1, 65):
        with pytest.raises(LobsimError):
            sim.book_depth(bad)
    pp, vp = ctypes.c_void_p(p.data_ptr()), ctypes.c_void_p(v.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = lib()
    assert L.lobsim_get_depth_dev(sim._h, 3, pp, vp, None, None, st) == abi.OK
    for depth, a, b in ((0, pp, vp), (65, pp, vp), (3, None, vp), (3, pp, None)):
        c = sim.launch_count
        assert L.lobsim_get_depth_dev(sim._h, depth, a, b, None, None, st) == abi.E_INVALID, depth
        assert sim.launch_count == c
    assert L.lobsim_get_depth_dev(None, 3, pp, vp, None, None, st) == abi.E_INVALID
    with pytest.raises(ValueError):
        sim.book_depth(3, out=(p, v.to(torch.int32)))
    sim.close()
