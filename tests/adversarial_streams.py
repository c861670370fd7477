"""Seeded adversarial packed streams for the replay kernels (CPU only).

The synthetic generator (csrc/synth_lobster.cpp) and the MSFT fixture are self-consistent LOBSTER flow: limits never cross,
an execution takes at most the head order, a cancel never exceeds the order it names.  The streams built here mix ordinary
flow with every order class those streams leave out: crossing limits (filled, resting, walking levels, emptying a side),
market orders that fill several orders and levels or end exactly on an order boundary, over-size and unknown-id removals,
removals from the middle of long queues before the level is executed, limits inside the spread and far behind the touch,
flat order pools that are exactly full when a crossing limit arrives, hybrid hot pools that run empty inside one message,
a best level longer than the hybrid pool, extreme prices and volumes, EmptyOrderbookError in the middle of a second, and a
market order that takes exactly the whole opposite side.

Each stream is built message by message against an oracle book (resync off): the oracle only aims the messages, the
semantics under test are whatever the oracle does at replay time.  One shadow oracle per replay start (a book reset from
that second's snapshot) lets the builder aim at the books the replay really holds, e.g. an EmptyOrderbookError that kills
some of the replayed books only.  Snapshots are the aimed book at every second boundary.

``classify`` counts the message classes through the oracle, message by message after ``reset_book``, resync ignored."""
from __future__ import annotations

import functools

import numpy as np

from rl4mm_b200 import abi
from rl4mm_b200.packing import PackedStream

SPS = 10                  # grid steps per second (100 ms grid)
HYB_CAP = 128             # orders in the hot pool of one side of the hybrid book (csrc/book_hybrid.cuh)
N_SECONDS = 64
STARTS = (0, 7, 16, 27, 41, 49)          # replay starts (seconds) the streams are aimed at
D_SECOND, KILL_SECOND = 34, 58           # a large order far behind the bid touch; the market order that kills some books
EMPTY_SIDE_SECONDS = ((10, abi.SELL), (22, abi.BUY), (45, abi.SELL))   # a crossing limit empties this side, then an exact sweep
HYB_SECONDS = (12, 18, 30, 38, 52)       # deep streams: sweeps through the hot pool, a level longer than the pool

# shape -> snapshot levels, capacity triple (levels, orders, agent orders per side), seeds
SHAPES = {
    "thin": dict(n_levels=10, caps=(64, 256, 32), seeds=(0, 1)),            # flat order pools (k_replay_flat)
    "deep": dict(n_levels=50, caps=(128, 1024, 64), seeds=(0, 1)),          # hybrid book (k_replay_hyb); 128/512 also fits
    "untemplated": dict(n_levels=20, caps=(96, 384, 32), seeds=(0,)),       # no compiled layout: the general kernel
}

CLASSES = (
    "cross_full", "cross_rest", "cross_walk", "cross_empty_side",
    "mkt_multi_order", "mkt_multi_level", "mkt_order_boundary", "mkt_leave_one", "mkt_exact_side", "death",
    "cancel_partial", "cancel_exact", "cancel_oversize", "delete_partial", "delete_exact", "delete_oversize",
    "unknown_agg_partial", "unknown_agg_oversize", "unknown_no_level", "wrong_price", "reused_ref",
    "churn_exec", "inside_spread", "far_behind",
    "flat_full_cross", "hyb_sweep", "hyb_cross_rest", "hyb_long_level",
)
# classes that only some shapes aim at
SHAPE_CLASSES = {"thin": ("flat_full_cross",), "deep": ("hyb_sweep", "hyb_cross_rest", "hyb_long_level")}


def params(shape: str, seed: int) -> dict:
    p = dict(tick=100, mid=1_000_000, whale=False, target=50, max_levels=30, flat_cap=0, hybrid=False, rate=40, max_depth=12,
             far=True, d_order=True, empty_sides=EMPTY_SIDE_SECONDS)
    if shape == "thin":
        p.update(target=40, max_levels=26, flat_cap=64)
        if seed == 1:
            # a mid of 15 ticks: the bid side lives a few ticks above 0, so nothing rests far behind the touch (no room behind the
            # bids; far asks would lift the mid when the ask side is swept), and only the ask side is swept
            p.update(mid=1_500, max_depth=3, far=False, d_order=False, empty_sides=tuple((t, abi.SELL) for t, _ in EMPTY_SIDE_SECONDS))
    elif shape == "deep":
        p.update(target=200, max_levels=80, hybrid=True, rate=45)
        if seed == 1:
            p.update(whale=True)                                  # single volumes up to 1e9
    else:
        p.update(target=90, max_levels=45, mid=(1 << 30) + 123_400)   # prices >= 2^30
    return p


def cfg_for(shape: str, n_envs: int = 1, **kw) -> abi.Cfg:
    sh = SHAPES[shape]
    nl, no, na = sh["caps"]
    base = dict(n_levels=sh["n_levels"], max_levels_per_side=nl, max_orders_per_side=no, max_agent_orders=na)
    base.update(kw)
    return abi.default_cfg(n_envs=n_envs, **base)


def _oracle(n_levels: int):
    from oracle.oracle import Oracle

    return Oracle(abi.default_cfg(n_levels=n_levels, resync=0, max_levels_per_side=4096, max_orders_per_side=1 << 20))


def _levels(entries: np.ndarray):
    """dump_book entries -> [(price, [(ref, volume), ...]), ...] best level first, FIFO inside a level."""
    out = []
    for p, r, v in zip(entries["price"].tolist(), entries["ref"].tolist(), entries["volume"].tolist()):
        if not out or out[-1][0] != p:
            out.append((p, []))
        out[-1][1].append((r, v))
    return out


class _Builder:
    def __init__(self, shape: str, seed: int):
        sh = SHAPES[shape]
        self.shape, self.L = shape, sh["n_levels"]
        self.p = params(shape, seed)
        self.tick = self.p["tick"]
        self.rng = np.random.default_rng(4242 + 17 * seed + {"thin": 0, "deep": 1000, "untemplated": 2000}[shape])
        self.main = _oracle(self.L)
        self.shadows = {}                                         # start second -> oracle reset from that snapshot
        self.msgs, self.step_off, self.snaps = [], [0], []
        self.next_ref = 1
        self.used_refs = set()
        self.reusable = []                                        # refs whose order left every replayed book for good
        self._cache = [None, None]
        self.second = 0
        self.d_ref = None
        self.pending_deletes = []                                 # (side, ref) of the orders that filled a flat pool
        tk, mid = self.tick, self.p["mid"]
        book = []
        for side in (abi.BUY, abi.SELL):
            n = min(self.L + 4, (mid // tk - 1) if side == abi.BUY else self.L + 4)
            ent = [(mid + (tk if side else -tk) * (k + 1), int(self.rng.integers(20, 300)), abi.REF_AGGREGATE, k) for k in range(n)]
            book.append(np.array(ent, abi.BOOK_ENTRY_DTYPE))
        self.main.set_book(book[0], book[1])

    # ---- the aimed book ---------------------------------------------------------------------------------------------
    def side(self, s: int):
        if self._cache[s] is None:
            self._cache[s] = _levels(self.main.dump_book(s))
        return self._cache[s]

    def best(self, s: int):
        lv = self.side(s)
        return lv[0][0] if lv else None

    def n_orders(self, s: int) -> int:
        return sum(len(q) for _, q in self.side(s))

    def total(self, s: int) -> int:
        return sum(v for _, q in self.side(s) for _, v in q)

    def fresh_ref(self) -> int:
        r = self.next_ref
        self.next_ref += 1
        return r

    def emit(self, mtype: int, s: int, price: int, vol: int, ref: int):
        assert 0 < vol < 2**31 and (mtype == abi.MSG_MARKET or 0 < price < 2**31 - 1), (mtype, price, vol)
        self.msgs.append((price, vol, ref, abi.meta(mtype, s)))
        self.main.process_order(mtype, s, price, vol, 1, ref)
        for o in self.shadows.values():
            o.process_order(mtype, s, price, vol, 1, ref)
        self._cache = [None, None]
        if mtype == abi.MSG_LIMIT:
            self.used_refs.add(ref)

    @property
    def live_refs(self) -> set:
        """refs that name a resting order of the aimed book"""
        return {r for side in (0, 1) for _, q in self.side(side) for r, _ in q if r != abi.REF_AGGREGATE}

    # ---- message kinds ----------------------------------------------------------------------------------------------
    def limit_price(self, s: int, depth: int):
        """A non-crossing limit price ``depth`` ticks behind the own best (or behind the opposite best when the side is empty)."""
        tk, b, o = self.tick, self.best(s), self.best(s ^ 1)
        if b is None:
            b = (o - tk) if (o is not None and s == abi.BUY) else (o + tk if o is not None else self.p["mid"])
        p = b - depth * tk if s == abi.BUY else b + depth * tk
        if o is not None and (p >= o if s == abi.BUY else p <= o):
            p = o - tk if s == abi.BUY else o + tk
        return p if p >= tk else None

    def vol(self, hi=200) -> int:
        if self.p["whale"] and self.rng.random() < 0.004 and max(self.total(0), self.total(1)) < 200_000_000:
            return int(self.rng.integers(100_000_000, 1_000_000_001))      # <= 1e9; every side stays below 2^31 in total
        return int(np.clip(np.exp(self.rng.normal(3.2, 1.0)), 1, hi))

    def rest(self, s: int, depth=None):
        if depth is None:
            depth = int(min(self.rng.geometric(0.25) - 1, 30 if self.p["hybrid"] else self.p["max_depth"]))
        p = self.limit_price(s, depth)
        if p is None or (len(self.side(s)) >= self.p["max_levels"] and all(lp != p for lp, _ in self.side(s))):
            p = self.best(s)
            if p is None:
                return
        ref = self.fresh_ref()
        self.emit(abi.MSG_LIMIT, s, p, self.vol(), ref)

    def reuse(self, s: int):
        if not self.reusable:
            return
        ref = self.reusable.pop(0)
        p = self.limit_price(s, int(self.rng.integers(0, 4)))
        if p is not None:
            self.emit(abi.MSG_LIMIT, s, p, self.vol(), ref)

    def inside_spread(self, s: int):
        b, o = self.best(s), self.best(s ^ 1)
        if b is None or o is None or abs(o - b) < 2 * self.tick:
            return
        p = b + self.tick if s == abi.BUY else b - self.tick
        self.emit(abi.MSG_LIMIT, s, p, self.vol(), self.fresh_ref())

    def far_behind(self, s: int, vol=None, ref=None, force=False):
        lv = self.side(s)
        if not self.p["far"] or not lv or (len(lv) >= self.p["max_levels"] - 2 and not force):
            return None
        worst = lv[-1][0]
        p = lv[0][0] + (-1 if s == abi.BUY else 1) * self.tick * int(self.rng.integers(100, 140))
        p = min(p, worst - self.tick) if s == abi.BUY else max(p, worst + self.tick)
        if p < self.tick:
            return None
        ref = self.fresh_ref() if ref is None else ref
        self.emit(abi.MSG_LIMIT, s, p, self.vol() if vol is None else vol, ref)
        return ref

    def remove_live(self, s: int, mode: str):
        cands = [(p, r, v) for p, q in self.side(s) for r, v in q if r != abi.REF_AGGREGATE and r != self.d_ref]
        if not cands:
            return
        p, r, v = cands[int(self.rng.integers(len(cands)))]
        if mode == "partial" and v < 2:
            mode = "exact"
        rv = int(self.rng.integers(1, v)) if mode == "partial" else v if mode == "exact" else v + int(self.rng.integers(1, 50))
        t = abi.MSG_CANCEL if self.rng.random() < 0.5 else abi.MSG_DELETE
        self.emit(t, s, p, rv, r)

    def remove_unknown_aggregate(self, s: int, over: bool):
        lv = [(p, q[0][1]) for p, q in self.side(s) if q[0][0] == abi.REF_AGGREGATE]
        if not lv:
            return
        p, v = lv[int(self.rng.integers(len(lv)))]
        if not over and v < 2:
            return
        rv = v + int(self.rng.integers(0, 30)) if over else int(self.rng.integers(1, v))
        self.emit(abi.MSG_CANCEL if self.rng.random() < 0.5 else abi.MSG_DELETE, s, p, rv, self.fresh_ref())

    def remove_no_level(self, s: int):
        b = self.best(s)
        if b is None:
            return
        prices = {p for p, _ in self.side(s)}
        for k in range(1, 40):
            p = b - k * self.tick if s == abi.BUY else b + k * self.tick
            if p >= self.tick and p not in prices:
                r = int(self.rng.choice(sorted(self.live_refs))) if self.live_refs and self.rng.random() < 0.5 else self.fresh_ref()
                self.emit(abi.MSG_DELETE, s, p, self.vol(), r)
                return

    def wrong_price(self, s: int):
        lv = self.side(s)
        cands = [(p, r) for p, q in lv for r, _ in q if r != abi.REF_AGGREGATE and r != self.d_ref]
        if len(lv) < 2 or not cands:
            return
        p, r = cands[int(self.rng.integers(len(cands)))]
        other = [lp for lp, _ in lv if lp != p]
        self.emit(abi.MSG_CANCEL, s, int(self.rng.choice(other)), self.vol(), r)

    def stale_remove(self, s: int):
        dead = sorted(self.used_refs - self.live_refs)
        b = self.best(s)
        if dead and b is not None:
            self.emit(abi.MSG_DELETE, s, b, self.vol(), int(self.rng.choice(dead)))

    def _fifo(self, s: int, max_orders=10**9):
        """[(price, volume, level index)] of the opposite-side orders an aggressor of side s meets, in execution order."""
        out = []
        for li, (p, q) in enumerate(self.side(s ^ 1)):
            for _, v in q:
                out.append((p, v, li))
                if len(out) >= max_orders:
                    return out
        return out

    def market(self, s: int, kind: str):
        fifo = self._fifo(s, 400)
        if len(fifo) < 3:
            return
        cum = np.cumsum([v for _, v, _ in fifo])
        if kind == "head":
            v = int(self.rng.integers(1, fifo[0][1] + 1))
        elif kind == "orders":        # several orders, ending exactly on an order boundary, or leaving 1 share at the head
            k = int(self.rng.integers(2, min(6, len(fifo) - 1) + 1))
            v = int(cum[k - 1]) - (1 if self.rng.random() < 0.4 and fifo[k - 1][1] > 1 else 0)
        else:                         # several levels
            lvl = int(self.rng.integers(1, 5))
            idx = [i for i, f in enumerate(fifo) if f[2] <= lvl]
            v = int(cum[idx[-1]]) - int(self.rng.integers(0, max(fifo[idx[-1]][1], 1)))
        if v >= int(cum[-1]) or v > self.total(s ^ 1) // 2 + 1:
            return
        self.emit(abi.MSG_MARKET, s, 0, max(v, 1), 0)

    def cross(self, s: int):
        opp = self.side(s ^ 1)
        if len(opp) < 3:
            return
        walk = int(self.rng.integers(0, min(5, len(opp) - 1)))      # levels crossed beyond the best
        p = opp[walk][0]
        avail = sum(v for _, q in opp[: walk + 1] for _, v in q)
        u = self.rng.random()
        v = int(self.rng.integers(1, avail + 1)) if u < 0.5 else avail + int(self.rng.integers(1, 100))
        if avail > self.total(s ^ 1) // 2 + 1:
            return
        self.emit(abi.MSG_LIMIT, s, p, v, self.fresh_ref())

    # ---- scripted sequences -----------------------------------------------------------------------------------------
    def churn(self):
        """A new best level of >= 6 orders, two removed from the middle of its queue, then a market order through it."""
        s = int(self.rng.integers(2))
        b, o = self.best(s), self.best(s ^ 1)
        if b is None or o is None:
            return
        p = b + self.tick if s == abi.BUY else b - self.tick
        if p <= 0 or (p >= o if s == abi.BUY else p <= o):
            p = b
        refs = []
        for _ in range(int(self.rng.integers(6, 9))):
            r = self.fresh_ref()
            self.emit(abi.MSG_LIMIT, s, p, int(self.rng.integers(1, 60)), r)
            refs.append(r)
        for r in (refs[2], refs[4]):
            t = abi.MSG_DELETE if self.rng.random() < 0.5 else abi.MSG_CANCEL
            vol = dict(q for lp, qq in self.side(s) if lp == p for q in qq).get(r, 0)
            if vol:
                self.emit(t, s, p, vol, r)
                self.reusable.append(r)                           # placed and removed in full inside one second
        fifo = self._fifo(s ^ 1)
        cum = np.cumsum([v for _, v, _ in fifo])
        at = [i for i, f in enumerate(fifo) if f[0] == p]
        if len(at) >= 3:
            k = at[min(len(at) - 1, int(self.rng.integers(2, 5)))]
            self.emit(abi.MSG_MARKET, s ^ 1, 0, int(cum[k]) - int(self.rng.integers(0, 2)), 0)

    def flat_full(self, start: int, s: int):
        """At the first message of second `start`: the flat pool of side s in the book replayed from `start` becomes exactly full,
        then a crossing limit of side s arrives (the flat path must hand the book to the sorted form before executing)."""
        cap = self.p["flat_cap"]
        sh = self.shadows[start]
        n = len(sh.dump_book(s))
        refs = []
        for _ in range(cap - n):
            r = self.fresh_ref()
            self.emit(abi.MSG_LIMIT, s, self.limit_price(s, int(self.rng.integers(0, 6))), int(self.rng.integers(1, 30)), r)
            refs.append(r)
        assert len(sh.dump_book(s)) == cap
        opp = self.side(s ^ 1)
        self.emit(abi.MSG_LIMIT, s, opp[min(1, len(opp) - 1)][0], sum(v for _, v in opp[0][1]) + int(self.rng.integers(1, 40)), self.fresh_ref())
        return refs

    def empty_side(self, s_opp: int):
        """A crossing limit takes the whole of side s_opp and rests; a few new orders there; a market order takes exactly all of
        them (no error); the side is rebuilt."""
        s = s_opp ^ 1
        opp = self.side(s_opp)
        if not opp:
            return
        tot = max(self.total(s_opp), *(self._shadow_total(o, s_opp) for o in self.shadows.values()))
        self.emit(abi.MSG_LIMIT, s, opp[-1][0], tot + int(self.rng.integers(1, 80)), self.fresh_ref())
        b = self.best(s)
        tot = 0
        for k in range(int(self.rng.integers(3, 7))):
            v = int(self.rng.integers(1, 80))
            p = b + self.tick * (1 + k // 2) if s_opp == abi.SELL else b - self.tick * (1 + k // 2)
            if p < self.tick:
                break
            self.emit(abi.MSG_LIMIT, s_opp, p, v, self.fresh_ref())
            tot += v
        if tot:
            self.emit(abi.MSG_MARKET, s, 0, tot, 0)
        for _ in range(3 * self.L):
            self.rest(s_opp, int(self.rng.integers(1, min(2 * self.L, self.p["max_depth"] + 1))))

    @staticmethod
    def _shadow_total(o, s):
        d = o.dump_book(s)
        return int(d["volume"].sum()) if len(d) else 0

    def hyb_sweep(self, s: int, rest: bool):
        """An execution of more than HYB_CAP orders in one message (the hot pool runs empty and is refilled while it lasts); with
        `rest`, a crossing limit whose remainder rests after the refills."""
        fifo = self._fifo(s, 1000)
        if len(fifo) < HYB_CAP + 40:
            return
        hi = min(len(fifo) * 6 // 10, HYB_CAP + 120)
        if hi < HYB_CAP + 5:
            return
        k = int(self.rng.integers(HYB_CAP + 5, hi + 1))
        cum = int(sum(v for _, v, _ in fifo[:k]))
        if rest:
            li = fifo[k - 1][2]
            p = self.side(s ^ 1)[li][0]
            avail = sum(v for _, v, l in fifo if l <= li)
            self.emit(abi.MSG_LIMIT, s, p, avail + int(self.rng.integers(1, 200)), self.fresh_ref())
        else:
            self.emit(abi.MSG_MARKET, s, 0, cum - int(self.rng.integers(0, 2)), 0)
        for _ in range(k):
            self.rest(s ^ 1)

    def long_level(self, s: int):
        """A level of more than HYB_CAP orders two ticks behind the best of side s, then a market order that ends inside it."""
        b = self.best(s)
        if b is None:
            return
        p = b - 2 * self.tick if s == abi.BUY else b + 2 * self.tick
        refs = []
        for _ in range(HYB_CAP + int(self.rng.integers(5, 20))):
            r = self.fresh_ref()
            self.emit(abi.MSG_LIMIT, s, p, int(self.rng.integers(1, 6)), r)
            refs.append(r)
        fifo = self._fifo(s ^ 1)
        at = [i for i, f in enumerate(fifo) if f[0] == p]
        k = at[int(self.rng.integers(2, 30))]
        self.emit(abi.MSG_MARKET, s ^ 1, 0, int(np.sum([v for _, v, _ in fifo[: k + 1]])), 0)
        for r in refs:                                             # the rest of the long level leaves again
            if r in self.live_refs:
                self.emit(abi.MSG_DELETE, s, p, 10, r)

    def kill(self):
        """A market sell in the middle of a second that empties the bid side of some replayed books (EmptyOrderbookError) and not
        of others: one more share than the smallest bid side among the replayed books (all of them when their bid sides hold
        the same volume)."""
        tots = [self._shadow_total(o, abi.BUY) for o in self.shadows.values() if not (o.state()["err"] & abi.ERR_EMPTY_BOOK)]
        asks = self.main.dump_book(abi.SELL)
        self.emit(abi.MSG_MARKET, abi.SELL, 0, min(tots) + 1, 0)
        if self.main.state()["err"] & abi.ERR_EMPTY_BOOK:         # the aimed book died too: it goes on with the asks it had
            self.main.set_book(np.zeros(0, abi.BOOK_ENTRY_DTYPE), asks)
            self._cache = [None, None]
        for _ in range(3 * self.L):
            self.rest(abi.BUY, int(self.rng.integers(0, min(2 * self.L, self.p["max_depth"] + 1))))

    # ---- ordinary flow ----------------------------------------------------------------------------------------------
    def flow(self):
        rng = self.rng
        s = int(rng.integers(2))
        n_own = self.n_orders(s)
        lv = self.side(s)
        if len(lv) > self.p["max_levels"] or n_own > self.p["target"] * 1.6:     # the worst level gives way: capacities hold
            for p, q in reversed(lv):
                for r, v in q:
                    if r != self.d_ref:
                        return self.emit(abi.MSG_DELETE, s, p, v, r if r != abi.REF_AGGREGATE else self.fresh_ref())
        if n_own < self.p["target"] * 0.7 or not lv:
            return self.rest(s)
        u = rng.random()
        over = n_own > self.p["target"] * 1.3
        if u < (0.30 if over else 0.42):
            return self.rest(s)
        if u < 0.46:
            return self.inside_spread(s)
        if u < 0.475:
            return self.far_behind(s)
        if u < 0.70:
            return self.remove_live(s, str(rng.choice(["partial", "exact", "over"], p=[0.4, 0.35, 0.25])))
        if u < 0.73:
            return self.remove_unknown_aggregate(s, rng.random() < 0.5)
        if u < 0.745:
            return self.remove_no_level(s)
        if u < 0.76:
            return self.wrong_price(s)
        if u < 0.775:
            return self.stale_remove(s)
        if u < 0.785:
            return self.reuse(s)
        if self.n_orders(s ^ 1) < self.p["target"] * 0.6:
            return self.rest(s ^ 1)
        if u < 0.90:
            return self.market(s, str(rng.choice(["head", "orders", "levels"])))
        return self.cross(s)

    # ---- the stream -------------------------------------------------------------------------------------------------
    def snapshot(self):
        row = np.zeros((2, self.L, 2), np.int32)
        row[..., 0] = abi.NO_PRICE
        for s in (0, 1):
            for k, (p, q) in enumerate(self.side(s)[: self.L]):
                row[s, k] = (p, sum(v for _, v in q))
        self.snaps.append(row)
        return row

    def build(self) -> PackedStream:
        rng = self.rng
        for sec in range(N_SECONDS):
            self.second = sec
            row = self.snapshot()
            if sec in STARTS:                                      # the book a replay from this second starts with
                o = _oracle(self.L)
                ent = []
                for s in (0, 1):
                    e = [(int(p), int(v), abi.REF_AGGREGATE, k) for k, (p, v) in enumerate(row[s]) if p != abi.NO_PRICE]
                    ent.append(np.array(e, abi.BOOK_ENTRY_DTYPE))
                o.set_book(ent[0], ent[1])
                self.shadows[sec] = o
            for st in range(SPS):
                if st == 0 and sec in STARTS and self.p["flat_cap"]:
                    refs = self.flat_full(sec, sec // 7 % 2)
                    self.pending_deletes = [(sec // 7 % 2, r) for r in refs]
                if st == 2 and sec % 3 == 1:
                    self.churn()
                if st == 4 and sec in dict(self.p["empty_sides"]):
                    self.empty_side(dict(self.p["empty_sides"])[sec])
                if st == 6 and sec == D_SECOND and self.p["d_order"]:
                    self.d_ref = self.far_behind(abi.BUY, vol=10**9 if self.p["whale"] else 10**6, force=True)
                    assert self.d_ref is not None
                if st == 5 and sec == KILL_SECOND:
                    self.kill()
                if self.p["hybrid"] and st == 3 and sec in HYB_SECONDS:
                    k = HYB_SECONDS.index(sec)
                    if k % 2 == 0:
                        self.hyb_sweep(k // 2 % 2, rest=k % 4 == 2)
                    else:
                        self.long_level(k // 2 % 2)
                if self.p["hybrid"] and st == 7 and sec in HYB_SECONDS:
                    self.hyb_sweep(1 - HYB_SECONDS.index(sec) % 2, rest=True)
                for _ in range(int(rng.poisson(self.p["rate"]))):
                    if self.pending_deletes and rng.random() < 0.3:
                        s, r = self.pending_deletes.pop()
                        for p, q in self.side(s):
                            if any(rr == r for rr, _ in q):
                                self.emit(abi.MSG_DELETE, s, p, 10**6, r)
                                break
                        continue
                    self.flow()
                self.step_off.append(len(self.msgs))
        self.snapshot()
        msgs = np.array(self.msgs, abi.MSG_DTYPE)
        snaps = np.array(self.snaps, np.int32)
        s = PackedStream(msgs, np.array(self.step_off, np.uint32), snaps, np.ones(len(snaps), np.uint8), 0, 100_000, self.L)
        s.validate()
        s.tick = self.tick
        return s


@functools.lru_cache(maxsize=None)
def build(shape: str, seed: int) -> PackedStream:
    """The seeded adversarial stream of one shape: N_SECONDS seconds, aimed at replays from the seconds of STARTS."""
    return _Builder(shape, seed).build()


# ---- classification ---------------------------------------------------------------------------------------------------
def classify(stream: PackedStream, cfg: abi.Cfg, start: int, n_steps: int) -> dict:
    """Counts of the message classes (CLASSES) a replay of ``n_steps`` grid steps from grid step ``start`` meets, message by
    message through the oracle: ``process_order`` after ``reset_book``, resync ignored.  ``cfg.tick_size`` is the tick of
    "far behind the touch" (100 ticks)."""
    from oracle.oracle import Oracle

    o = Oracle(abi.default_cfg(n_levels=stream.n_levels, resync=0, tick_size=cfg.tick_size), stream)
    o.reset_book(start)
    flat_cap = 32 * (4 if cfg.max_levels_per_side >= 128 and cfg.max_orders_per_side >= 256 else 2)
    c = dict.fromkeys(CLASSES, 0)
    books = [_levels(o.dump_book(0)), _levels(o.dump_book(1))]
    used = set()
    churned = {0: set(), 1: set()}
    m0, m1 = int(stream.step_off[start]), int(stream.step_off[min(start + n_steps, stream.n_grid_steps)])
    for m in stream.msgs[m0:m1]:
        price, vol, ref, meta = int(m["price"]), int(m["volume"]), int(m["ref"]), int(m["meta"])
        t, s = meta & 7, (meta >> 3) & 1
        own, opp = books[s], books[s ^ 1]
        live = {r: (p, v) for p, q in own for r, v in q if r != abi.REF_AGGREGATE}
        o.clear_fills()
        o.process_order(t, s, price, vol, 1, ref)
        fills = o.fills()                                         # (external aggressor: one record per resting order hit)
        after = list(books)
        for side in ((s,) if t != abi.MSG_MARKET and not len(fills) else (0, 1)):
            after[side] = _levels(o.dump_book(side))
        dead = bool(o.state()["err"] & abi.ERR_EMPTY_BOOK)
        if t in (abi.MSG_LIMIT, abi.MSG_MARKET):
            n_fill = len(fills)
            lv_prices = {int(f["price"]) for f in fills}
            if t == abi.MSG_LIMIT:
                if ref in used:
                    c["reused_ref"] += 1
                used.add(ref)
                if n_fill:
                    rested = sum(v for _, q in after[s] for r, v in q if r == ref)
                    c["cross_rest" if rested else "cross_full"] += 1
                    c["cross_walk"] += 2 <= len(lv_prices) <= 5
                    c["cross_empty_side"] += bool(rested and not after[s ^ 1])
                    if flat_cap and sum(len(q) for _, q in own) == flat_cap:
                        c["flat_full_cross"] += 1
                    c["hyb_cross_rest"] += bool(rested and n_fill > HYB_CAP)
                elif own and opp:
                    b, a = (own[0][0], opp[0][0])
                    c["inside_spread"] += (price > b) if s == abi.BUY else (price < b)
                    c["far_behind"] += (b - price if s == abi.BUY else price - b) >= 100 * cfg.tick_size
            else:
                if dead:
                    c["death"] += 1
                elif n_fill:
                    c["mkt_multi_order"] += n_fill >= 2 and len(lv_prices) < n_fill
                    c["mkt_multi_level"] += len(lv_prices) >= 2
                    c["mkt_exact_side"] += not after[s ^ 1]
                    if after[s ^ 1]:
                        nb = sum(len(q) for _, q in opp) - sum(len(q) for _, q in after[s ^ 1])
                        head_left = after[s ^ 1][0][1][0][1]
                        c["mkt_order_boundary"] += n_fill >= 2 and nb == n_fill
                        c["mkt_leave_one"] += n_fill >= 2 and nb == n_fill - 1 and head_left == 1
                    c["hyb_sweep"] += n_fill > HYB_CAP
            if n_fill >= 2:
                for p, q in opp:
                    if p in lv_prices and sum(1 for f in fills if int(f["price"]) == p) >= 2:
                        c["churn_exec"] += p in churned[s ^ 1]
                        c["hyb_long_level"] += len(q) > HYB_CAP
        else:
            kind = "cancel" if t == abi.MSG_CANCEL else "delete"
            lv = dict(own)
            if ref in live and live[ref][0] == price:
                v = live[ref][1]
                c[f"{kind}_{'partial' if vol < v else 'exact' if vol == v else 'oversize'}"] += 1
                q = lv[price]
                pos = [r for r, _ in q].index(ref)
                if len(q) >= 5 and 0 < pos < len(q) - 1:
                    churned[s].add(price)
            elif ref in live:
                c["wrong_price"] += 1
            elif price not in lv:
                c["unknown_no_level"] += 1
            elif lv[price][0][0] == abi.REF_AGGREGATE:
                c["unknown_agg_partial" if vol < lv[price][0][1] else "unknown_agg_oversize"] += 1
            if ref in used and ref not in live:
                c["reused_ref"] += 1
        for side in (0, 1):                                       # a level that disappears forgets its churn
            churned[side] &= {p for p, _ in after[side]}
        books = after
        if dead:
            break
    return c
