"""The adversarial streams of tests/adversarial_streams.py keep the coverage the GPU replay tests rely on: every message class
at least 5 times over the replays from the stream's start seconds (EmptyOrderbookError and the exact sweep of a whole side
at least once), valid packed streams, refs unique among resting orders, positive prices, and no capacity crossed."""
import numpy as np
import pytest

import adversarial_streams as A
from rl4mm_b200 import abi

STREAMS = [(shape, seed) for shape, sh in A.SHAPES.items() for seed in sh["seeds"]]
RARE = ("death", "mkt_exact_side")


def _minimum(shape, seed, cls):
    if cls in RARE:
        return 1
    for other, classes in A.SHAPE_CLASSES.items():
        if cls in classes and other != shape:
            return 0
    if cls == "far_behind" and not A.params(shape, seed)["far"]:
        return 0          # the low-mid stream: no room behind the bids, and far asks would lift the mid at the next sweep
    return 5


@pytest.mark.parametrize("shape,seed", STREAMS)
def test_adversarial_stream_covers_every_class(shape, seed):
    s = A.build(shape, seed)
    cfg = A.cfg_for(shape, tick_size=s.tick)
    total = dict.fromkeys(A.CLASSES, 0)
    survivors = 0
    for start in A.STARTS:
        c = A.classify(s, cfg, 10 * start, s.n_grid_steps - 10 * start)
        for k, v in c.items():
            total[k] += v
        survivors += c["death"] == 0
    print(f"\n{shape}/{seed}: {s.n_msgs} messages, {s.n_seconds} s; classes over starts {A.STARTS}: {total}")
    low = {k: v for k, v in total.items() if v < _minimum(shape, seed, k)}
    assert not low, low
    assert survivors > 0, "EmptyOrderbookError kills some of the replayed books only"


@pytest.mark.parametrize("shape,seed", STREAMS)
def test_adversarial_stream_is_well_formed(shape, seed):
    from oracle.oracle import Oracle

    s = A.build(shape, seed)
    s.validate()
    assert s.n_seconds >= 60 and 20_000 <= s.n_msgs <= 40_000
    assert np.all(s.snap_valid == 1)
    m = s.msgs
    t = m["meta"] & 7
    assert np.all(m["volume"] > 0)
    assert np.all(m["price"][t != abi.MSG_MARKET] > 0)
    snap_p = s.snapshots[..., 0]
    assert np.all((snap_p > 0) | (snap_p == abi.NO_PRICE))
    assert np.all(s.snapshots[..., 1][snap_p != abi.NO_PRICE] > 0)
    mid = (int(s.snapshots[0, 0, 0, 0]) + int(s.snapshots[0, 1, 0, 0])) // 2
    if (shape, seed) == ("thin", 1):
        assert mid < 20 * s.tick                      # a mid of a few ticks
    if shape == "untemplated":
        assert np.all(m["price"][t != abi.MSG_MARKET] >= 2**30)
    if (shape, seed) == ("deep", 1):
        assert m["volume"][t == abi.MSG_LIMIT].max() >= 900_000_000
    # from every start: a limit never names a resting order's ref, sides stay below 2^31 shares, and no capacity is crossed
    nl, no, _ = A.SHAPES[shape]["caps"]
    for start in A.STARTS:
        o = Oracle(abi.default_cfg(n_levels=s.n_levels, resync=0), s)
        o.reset_book(10 * start)
        seen = set()
        for step in range(10 * start, s.n_grid_steps):
            for i in range(int(s.step_off[step]), int(s.step_off[step + 1])):
                if (int(m["meta"][i]) & 7) == abi.MSG_LIMIT and int(m["ref"][i]) in seen:   # a reused ref
                    for side in (0, 1):
                        assert int(m["ref"][i]) not in o.dump_book(side)["ref"], (start, i)
                seen.add(int(m["ref"][i]))
                o.process_order(int(m["meta"][i]) & 7, (int(m["meta"][i]) >> 3) & 1, int(m["price"][i]), int(m["volume"][i]),
                                1, int(m["ref"][i]))
            if o.state()["err"]:
                break
            if step % 10 == 9:
                for side in (0, 1):
                    assert int(o.dump_book(side)["volume"].astype(np.int64).sum()) < 2**31
        p = o.peaks()
        assert max(p["levels"]) <= nl and max(p["orders"]) <= no and (shape != "deep" or max(p["orders"]) <= 512), (start, p)
