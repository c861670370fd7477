"""The replay kernels walk a launch one second at a time, not one grid step at a time: a replay book holds no agent orders, so
only second boundaries (resync, trackers, flat re-entry) are points where anything happens between messages.  These tests put
every boundary that such a loop creates next to the oracle: launches that start and end part-way through a second, steps and
whole seconds without messages, a stream that ends part-way through a second, a book that dies of EmptyOrderbookError in the
middle of a second (now_step must be the step of the fatal message), message tiles with non-positive volumes, and a flat order
pool that fills part-way through a second so that the book goes on in the sorted form inside a message segment."""
import numpy as np
import pytest

from rl4mm_b200 import abi
from rl4mm_b200.packing import PackedStream

pytestmark = [pytest.mark.gpu, pytest.mark.replay_path]

SPS = 10                 # steps per second at the default 100 ms grid
N_GRID = 57              # the stream ends part-way through its sixth second
EMPTY_SECOND = 3         # steps 30..39 carry no message
KILL_STEP = 23           # the market order that empties the bid side (in the middle of second 2, not its first message)
BURST_STEPS = (14, 45)   # 80 resting buy orders: more than the 64-order flat pool of the 64/256/32 layout
CAP = dict(max_levels_per_side=64, max_orders_per_side=256)


def _stream(seed: int, kill: bool, bad_volume: bool) -> PackedStream:
    rng = np.random.default_rng(seed)
    n_levels, tick = 10, 100
    n_sec = (N_GRID + SPS - 1) // SPS
    snaps = np.zeros((n_sec + 1, 2, n_levels, 2), np.int32)
    snaps[..., 0] = abi.NO_PRICE
    for lv in range(6):
        snaps[:, 0, lv] = (10_000 - tick * (lv + 1), 20 + 5 * lv)
        snaps[:, 1, lv] = (10_000 + tick * (lv + 1), 20 + 5 * lv)
    msgs, step_off, live, ref = [], [0], [], 1000

    def add(price, volume, r, mtype, side):
        msgs.append((price, volume, r, abi.meta(mtype, side)))

    for step in range(N_GRID):
        n = 0 if step // SPS == EMPTY_SECOND else int(rng.choice([0, 0, 1, 3, 7, 20, 45]))
        for j in range(n):
            u = rng.random()
            side = int(rng.integers(2))
            if u < 0.5 or not live:
                price = 10_000 + (tick if side else -tick) * int(rng.integers(0, 6))
                add(price, int(rng.integers(1, 40)), ref, abi.MSG_LIMIT, side)
                live.append((price, ref, side))
                ref += 1
            elif u < 0.9:
                price, r, s = live.pop(int(rng.integers(len(live))))
                add(price, int(rng.integers(1, 60)), r, abi.MSG_CANCEL if rng.random() < 0.3 else abi.MSG_DELETE, s)
            else:
                add(0, int(rng.integers(1, 25)), 0, abi.MSG_MARKET, side)
            if bad_volume and step in (5, 44) and j == 1:
                add(10_000 - tick, 0 if step == 5 else -3, ref, abi.MSG_LIMIT, abi.BUY)
                ref += 1
        if step in BURST_STEPS:
            for k in range(80):
                add(10_000 - tick * (1 + k % 5), 1 + k % 7, ref, abi.MSG_LIMIT, abi.BUY)
                live.append((10_000 - tick * (1 + k % 5), ref, abi.BUY))
                ref += 1
        if kill and step == KILL_STEP:
            add(10_000 - tick, 5, ref, abi.MSG_LIMIT, abi.BUY)
            ref += 1
            add(0, 10 ** 7, 0, abi.MSG_MARKET, abi.SELL)
            add(10_000 + tick, 5, ref, abi.MSG_LIMIT, abi.SELL)
            ref += 1
        step_off.append(len(msgs))
    m = np.array(msgs, abi.MSG_DTYPE)
    s = PackedStream(m, np.array(step_off, np.uint32), snaps, np.ones(n_sec + 1, np.uint8), 0, 100_000, n_levels)
    s.validate()
    return s


def _check(sim, oracles, what):
    from test_gpu_parity import compare_books

    st = sim.state()
    for env, o in enumerate(oracles):
        os_ = o.state()
        assert int(st["err"][env]) == int(os_["err"]), (what, env, int(st["err"][env]), int(os_["err"]))
        assert int(st["now_step"][env]) == int(os_["now_step"]), (what, env, int(st["now_step"][env]), int(os_["now_step"]))
        if int(os_["err"]) & abi.ERR_EMPTY_BOOK:
            continue   # the reference raises: the book of a dead env is left as it was when the error struck (not compared)
        for f in ("min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume"):
            assert st[f][env] == os_[f], (what, env, f, st[f][env], os_[f])
        compare_books(sim, env, o, (what, env))


@pytest.mark.parametrize("kill,bad_volume", [(False, False), (True, False), (False, True)])
def test_replay_boundaries_inside_seconds_match_oracle(kill, bad_volume):
    """Ragged launches (T not a multiple of the second, starting part-way through one) over a stream with empty steps, an empty
    second, a pool that overflows in the middle of a second and an end part-way through a second; optionally a book that dies in
    the middle of a second, or segments that carry non-positive volumes.  State, books, now_step and error bits as the oracle's."""
    import torch

    assert torch.cuda.is_available()
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    s = _stream(7, kill, bad_volume)
    starts = np.array([0, 10, 20, 40], np.int32)
    kw = dict(n_levels=s.n_levels, outer_levels=3, resync=1)
    sim = LobSim(abi.default_cfg(n_envs=len(starts), **kw, **CAP), 0)
    sim.load_stream(0, s)
    sim.reset_book(0, starts)
    oracles = [Oracle(abi.default_cfg(n_envs=1, **kw, **CAP), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    _check(sim, oracles, "reset")
    for chunk in (3, 1, 7, 12, 0, 25, 4, 9, 2):
        sim.replay(chunk)
        for o in oracles:
            o.replay(chunk)
        _check(sim, oracles, ("replay", chunk))
    st = sim.state()
    assert np.all(st["now_step"][: len(starts)] <= N_GRID)
    assert int(st["err"][3]) & abi.ERR_END_OF_STREAM and int(st["now_step"][3]) == N_GRID
    if kill:
        for env in range(3):
            assert int(st["err"][env]) & abi.ERR_EMPTY_BOOK and int(st["now_step"][env]) == KILL_STEP, env
    sim.close()


def test_forward_step_between_ragged_replays_matches_oracle():
    """`forward_step` (resync only at the end of the call) over several seconds, between replay launches that start and stop
    part-way through a second."""
    import torch

    assert torch.cuda.is_available()
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    s = _stream(11, False, False)
    starts = np.array([0, 10, 20], np.int32)
    kw = dict(n_levels=s.n_levels, outer_levels=3, resync=1)
    sim = LobSim(abi.default_cfg(n_envs=len(starts), **kw, **CAP), 0)
    sim.load_stream(0, s)
    sim.reset_book(0, starts)
    oracles = [Oracle(abi.default_cfg(n_envs=1, **kw, **CAP), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    for kind, chunk in (("replay", 4), ("forward", 23), ("replay", 6), ("forward", 3), ("replay", 11)):
        if kind == "replay":
            sim.replay(chunk)
        else:
            sim.forward_step(chunk)
        for o in oracles:
            o.replay(chunk) if kind == "replay" else o.forward_step(chunk)
        _check(sim, oracles, (kind, chunk))
    sim.close()
