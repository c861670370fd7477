"""CPU tests of the oracle's forward_step, set_book and capacity high-water marks (oracle/lob_oracle.c): the twins of
lobsim_forward_step, lobsim_set_book and the device's capacity flags that the GPU tests compare against."""
import numpy as np

from oracle.oracle import Oracle
from rl4mm_b200 import abi, synthetic


def _stream(seed=3, **kw):
    sc = synthetic.SynthConfig(seed=seed, n_msgs=30_000, duration_s=80, n_levels=10, mid0=1_000_000, p_limit=0.45, p_cancel=0.2,
                               p_delete=0.25, p_exec=0.1, geom_p=0.35, init_levels=14, mean_queue=3, target_orders=60,
                               max_offset_ticks=20, p_sweep=0.01)
    for k, v in kw.items():
        setattr(sc, k, v)
    return synthetic.generate(sc)


def _same(a: Oracle, b: Oracle, what="", fields=("now_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell",
                                                   "best_buy_volume", "best_sell_volume", "err")):
    for side in (0, 1):
        assert np.array_equal(a.dump_book(side), b.dump_book(side)), (what, side)
        assert np.array_equal(a.dump_agent_orders(side), b.dump_agent_orders(side)), (what, side)
    sa, sb = a.state(), b.state()
    for f in fields:
        assert sa[f] == sb[f], (what, f, sa[f], sb[f])


def test_forward_step_one_equals_replay_one():
    s = _stream()
    kw = dict(n_levels=10, outer_levels=8, resync=1)
    a, b = Oracle(abi.default_cfg(**kw), s), Oracle(abi.default_cfg(**kw), s)
    a.reset_book(20)
    b.reset_book(20)
    for t in range(300):
        a.replay(1)
        b.forward_step(1)
        assert np.array_equal(a.fills(), b.fills()), t
        _same(a, b, f"step {t}")


def test_forward_step_n_equals_replay_n_without_resync():
    s = _stream(seed=4)
    kw = dict(n_levels=10, outer_levels=8, resync=0)
    for n in (2, 7, 10, 57):
        a, b = Oracle(abi.default_cfg(**kw), s), Oracle(abi.default_cfg(**kw), s)
        a.reset_book(10)
        b.reset_book(10)
        for k in range(5):
            a.replay(n)
            b.forward_step(n)
            assert np.array_equal(a.fills(), b.fills()), (n, k)
            _same(a, b, f"n {n} call {k}")


def test_forward_step_resyncs_only_at_the_end():
    """With resync on, replay(n) runs update_outer_levels at every whole second it crosses; forward_step(n) only at `until`.
    A thin book that leaves its initial price range within seconds makes the two differ; at n = 1 they never do."""
    s = _stream(seed=5, target_orders=20, init_levels=11, p_sweep=0.03)
    kw = dict(n_levels=10, outer_levels=9, resync=1)
    differs = 0
    for start in range(0, 400, 40):
        a, b = Oracle(abi.default_cfg(**kw), s), Oracle(abi.default_cfg(**kw), s)
        a.reset_book(start)
        b.reset_book(start)
        a.replay(30)              # crosses the seconds start+10 and start+20, ends on start+30
        b.forward_step(30)
        assert a.state()["now_step"] == b.state()["now_step"] == start + 30
        differs += any(not np.array_equal(a.dump_book(side), b.dump_book(side)) for side in (0, 1)) or \
            a.state()["min_buy_price"] != b.state()["min_buy_price"] or a.state()["max_sell_price"] != b.state()["max_sell_price"]
    assert differs >= 1


def _agent_book(seed=6):
    """An oracle at a replayed book with resting agent orders on both sides."""
    s = _stream(seed=seed)
    o = Oracle(abi.default_cfg(n_levels=10, outer_levels=8, resync=1), s)
    o.reset_book(30)
    o.replay(40)
    st = o.state()
    ids = []
    for k in range(6):
        side = k % 2
        px = int(st["best_buy"]) - 100 * (k // 2) if side == 0 else int(st["best_sell"]) + 100 * (k // 2)
        ids.append(o.process_order(abi.MSG_LIMIT, side, px, 7 + k, False, 0))
    o.replay(5)
    return s, o, ids


def test_set_book_round_trip_with_agent_orders():
    s, src, _ = _agent_book()
    buy, sell = src.dump_book(0), src.dump_book(1)
    assert ((buy["ref"] & abi.REF_AGENT) != 0).any() and ((sell["ref"] & abi.REF_AGENT) != 0).any()
    dst = Oracle(abi.default_cfg(n_levels=10, outer_levels=8, resync=1), s)
    dst.reset_book(300)                       # another clock: set_book leaves it where it is
    dst.process_order(abi.MSG_DELETE, 0, 1, 5, True, 1)   # an unknown-price delete: no-op
    st0 = dst.state()
    dst.set_book(buy, sell)
    for side in (0, 1):
        assert np.array_equal(dst.dump_book(side), src.dump_book(side)), side
        assert np.array_equal(dst.dump_agent_orders(side), src.dump_agent_orders(side)), side
    st = dst.state()
    assert st["now_step"] == st0["now_step"] and st["min_buy_price"] == st0["min_buy_price"]
    assert st["err"] == 0 and st["next_agent_id"] >= max(int(r) & 0x7fffffff for r in np.concatenate([buy["ref"], sell["ref"]])
                                                        if int(r) & abi.REF_AGENT)
    assert tuple(st["n_agent_orders"]) == tuple(src.state()["n_agent_orders"])


def test_set_book_then_orders_behave_like_the_source_book():
    """The rebuilt external-id map and internal ids: cancels, deletes, executions and agent cancels hit the same orders."""
    s, src, ids = _agent_book(seed=7)
    dst = Oracle(abi.default_cfg(n_levels=10, outer_levels=8, resync=1), s)
    dst.reset_book(300)
    dst.set_book(src.dump_book(0), src.dump_book(1))
    for side in (0, 1):                       # cancel one external order of each side by its external id, partially
        ext = [e for e in src.dump_book(side) if e["ref"] != abi.REF_AGGREGATE and not e["ref"] & abi.REF_AGENT]
        e = ext[len(ext) // 2]
        for o in (src, dst):
            o.process_order(abi.MSG_CANCEL, side, int(e["price"]), max(1, int(e["volume"]) // 2), True, int(e["ref"]))
    agent = src.dump_agent_orders(1)[0]
    for o in (src, dst):
        o.process_order(abi.MSG_CANCEL, 1, int(agent["price"]), int(agent["volume"]), False, int(agent["ref"]))
        o.clear_fills()
        o.process_order(abi.MSG_MARKET, 0, 0, 300, True, 0)
    assert np.array_equal(src.fills(), dst.fills())
    _same(src, dst, "after orders", fields=("best_buy", "best_sell", "best_buy_volume", "best_sell_volume", "err"))
    # the agent id counter of dst is above every id it was given: new agent orders get fresh ids
    new_id = dst.process_order(abi.MSG_LIMIT, 0, int(dst.state()["best_buy"]) - 1000, 5, False, 0)
    assert new_id > max(ids)


def test_set_book_rejects_an_unsorted_side_and_keeps_the_book():
    s, src, _ = _agent_book(seed=8)
    buy = src.dump_book(0)
    before = src.dump_book(1)
    bad = buy[::-1].copy()
    try:
        src.set_book(bad, before)
        raised = False
    except RuntimeError:
        raised = True
    assert raised and np.array_equal(src.dump_book(0), buy) and np.array_equal(src.dump_book(1), before)


def test_set_book_clears_the_error_bits():
    s = _stream(seed=9)
    o = Oracle(abi.default_cfg(n_levels=10), s)
    o.reset_book(10)
    o.process_order(abi.MSG_LIMIT, 0, 900_000, 0, True, 5)        # volume 0: BAD_VOLUME
    assert o.state()["err"] & abi.ERR_BAD_VOLUME
    o.set_book(o.dump_book(0), o.dump_book(1))
    assert o.state()["err"] == 0


def _counts(o: Oracle):
    lv = tuple(len(np.unique(o.dump_book(side)["price"])) for side in (0, 1))
    return lv, tuple(len(o.dump_book(side)) for side in (0, 1)), tuple(len(o.dump_agent_orders(side)) for side in (0, 1))


def test_peaks_are_monotone_upper_bounds_and_reset_by_reset_book():
    s, o, _ = _agent_book(seed=10)
    prev = o.peaks()
    for t in range(120):
        if t % 15 == 7:
            st = o.state()
            o.process_order(abi.MSG_LIMIT, t % 2, int(st["best_buy"]) - 300 if t % 2 == 0 else int(st["best_sell"]) + 300, 9, False, 0)
        o.replay(3)
        p = o.peaks()
        lv, nord, nag = _counts(o)
        for side in (0, 1):
            assert p["levels"][side] >= max(prev["levels"][side], lv[side])
            assert p["orders"][side] >= max(prev["orders"][side], nord[side])
            assert p["agents"][side] >= max(prev["agents"][side], nag[side])
        assert p["fills"] >= max(prev["fills"], len(o.fills()))
        prev = p
    assert max(prev["orders"]) > max(_counts(o)[1]) or max(prev["levels"]) >= max(_counts(o)[0])
    o.reset_book(100)
    p = o.peaks()
    lv, nord, nag = _counts(o)
    assert p == dict(levels=lv, orders=nord, agents=(0, 0), fills=0)


def test_peaks_count_the_book_at_its_largest():
    """A limit order that rests and is executed again in the same call still counts: the peak is the largest book, not the last."""
    s = _stream(seed=11)
    o = Oracle(abi.default_cfg(n_levels=10), s)
    o.reset_book(10)
    lv0, nord0, _ = _counts(o)
    bb = int(o.state()["best_buy"])
    for k in range(5):                        # five new buy levels below the book
        o.process_order(abi.MSG_LIMIT, 0, bb - 100 * (20 + k), 3, True, 1000 + k)
    for k in range(5):
        o.process_order(abi.MSG_DELETE, 0, bb - 100 * (20 + k), 3, True, 1000 + k)
    assert _counts(o)[0] == lv0
    p = o.peaks()
    assert p["levels"][0] == lv0[0] + 5 and p["orders"][0] == nord0[0] + 5
    o.clear_fills()
    o.replay(30)
    assert o.peaks()["fills"] == len(o.fills())
