"""lobsim_submit_orders_dev / LobSim.submit_orders: every env's own list of orders applied on the device in one launch.  Seeded
random order programs per env (limits that rest, cross, walk levels and meet the agent's own orders; market orders, one into an
empty side; cancels and deletes by agent id and external ref, partial, exact, over-size and volume None; unknown ids; bad
volumes; skipped types and directions) with ragged counts, against one oracle per env fed the same orders through
process_order: the L3 and agent books, state() field by field, the error bits, the fills in order and the refs.  Twin handles
show the call is bit-identical to lobsim_process_orders on the same orders.  Then: rows with count 0 and dead envs, the
portfolio and the handle's fill log, max_fills truncation, the capacity flags, flat blobs, env steps and rollouts after a
submission, the agent_orders -> submit_orders -> forward_step loop, CUDA graph capture, deep-book mode and the arguments."""
import ctypes

import numpy as np
import pytest

import adversarial_streams as A
import parity_helpers as H
from rl4mm_b200 import abi, synthetic

pytestmark = pytest.mark.gpu

FIELDS = ("inventory", "now_step", "episode_start_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume",
          "best_sell_volume", "err", "n_agent_orders")
KW = dict(n_levels=10, outer_levels=5, resync=1, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=64)
UNKNOWN_ID = 0x7FFFFFF0           # an agent id neither the device nor the oracle ever hands out
INT_MAX = 2**31 - 1


def _stream(seed=41, **kw):
    sc = dict(seed=seed, n_msgs=40_000, duration_s=100, n_levels=10, target_orders=80, p_sweep=0.02)
    sc.update(kw)
    return synthetic.generate(synthetic.SynthConfig(**sc))


def u32(t):
    return t.view(__import__("torch").int32).cpu().numpy().view(np.uint32)


def fills_of(fills, n_fills, env):
    f = fills.cpu().numpy()[env].copy().view(abi.FILL_DTYPE).reshape(-1)
    return f[: min(int(n_fills[env]), len(f))]


def pack(rows, K):
    import torch

    a = np.zeros((len(rows), K), abi.ORDER_DTYPE)
    for e, row in enumerate(rows):
        for i, (t, d, p, v, x, r) in enumerate(row):
            a[e, i] = (e, t, d, p, v, x, r & 0xFFFFFFFF, 0)
    return torch.from_numpy(a.view(np.int32).reshape(len(rows), K, 8).copy()).cuda()


class Bed:
    """A handle and one oracle per env on the same stream, started with reset_book (or reset) at `starts`."""

    def __init__(self, starts, s=None, env=False, **kw):
        from oracle.oracle import Oracle
        from test_gpu_parity import make_sim

        self.kw = dict(KW, **kw)
        self.s = s if s is not None else _stream()
        self.n = len(starts)
        self.cfg = abi.default_cfg(n_envs=self.n, **self.kw)
        self.sim = make_sim(self.cfg, [self.s])
        self.oracles = [Oracle(abi.default_cfg(**self.kw), self.s, env_index=i) for i in range(self.n)]
        starts = np.asarray(starts, np.int32)
        if env:
            self.sim.reset(0, starts)
        else:
            self.sim.reset_book(0, starts)
        for o, st in zip(self.oracles, starts):
            o.reset(int(st)) if env else o.reset_book(int(st))
        self.excluded = np.zeros(self.n, bool)
        self.ext_ref = 1 << 28
        self.stats = dict(rested=0, fills=0, bad_volume=0, empty_book=0, skipped=0)

    def replay(self, k):
        self.sim.replay(k)
        for o in self.oracles:
            o.replay(k)

    def forward_step(self, k):
        self.sim.forward_step(k)
        for o in self.oracles:
            o.forward_step(k)

    def id_map(self, env):
        """device agent id -> the oracle's internal id: the k-th agent order by id on both sides is the same order."""
        m = {}
        for side in (0, 1):
            d, o = self.sim.dump_agent_orders(env, side), self.oracles[env].dump_agent_orders(side)
            if len(d) == len(o):
                m.update(zip((d["ref"] & 0x7FFFFFFF).tolist(), (o["ref"] & 0x7FFFFFFF).tolist()))
        return m

    def program(self, rng, env, K, kinds=None):
        """A random order list for env, from its current books (device ids for the agent's orders)."""
        o = self.oracles[env]
        st = o.state()
        bb, bs = int(st["best_buy"]), int(st["best_sell"])
        if bb == 0 or bs == INT_MAX:
            return [(abi.MSG_LIMIT, 0, 1_000_000, 5, 0, 0)] * int(rng.integers(0, 3))      # a dead or one-sided book
        agents = [(side, int(e["price"]), int(e["volume"]), int(e["ref"]) & 0x7FFFFFFF) for side in (0, 1)
                  for e in self.sim.dump_agent_orders(env, side)]
        book = [(side, int(e["price"]), int(e["volume"]), int(e["ref"])) for side in (0, 1) for e in o.dump_book(side)]
        ext = [b for b in book if b[3] != abi.REF_AGGREGATE and not b[3] & abi.REF_AGENT]
        aggs = [b for b in book if b[3] == abi.REF_AGGREGATE]
        kinds = kinds or ["rest"] * 5 + ["cross"] * 2 + ["ext_limit"] * 2 + ["mkt", "ext_mkt"] + ["cancel_agent"] * 4 + \
            ["cancel_ext"] * 2 + ["unknown", "bad", "skip"]
        row = []
        for _ in range(int(rng.integers(0, K + 1))):
            kind = str(rng.choice(kinds))
            side = int(rng.integers(2))
            best, other = (bb, bs) if side == 0 else (bs, bb)
            sgn = -1 if side == 0 else 1                   # away from the touch
            if kind == "rest":
                row.append((abi.MSG_LIMIT, side, best + sgn * 100 * int(rng.integers(0, 5)), int(rng.integers(1, 80)), 0, 0))
            elif kind == "cross":                          # at or through the opposite best: fills, walks levels, self-matches
                row.append((abi.MSG_LIMIT, side, other - sgn * 100 * int(rng.integers(0, 3)), int(rng.integers(1, 300)), 0, 0))
            elif kind == "ext_limit":
                self.ext_ref += 1
                px = best + sgn * 100 * int(rng.integers(0, 4)) if rng.random() < 0.6 else other - sgn * 100 * int(rng.integers(0, 2))
                row.append((abi.MSG_LIMIT, side, px, int(rng.integers(1, 200)), 1, self.ext_ref))
            elif kind in ("mkt", "ext_mkt"):
                row.append((abi.MSG_MARKET, side, 0, int(rng.integers(1, 300)), int(kind == "ext_mkt"), 0))
            elif kind in ("cancel_agent", "cancel_ext"):
                pool = agents if kind == "cancel_agent" else ext
                if not pool:
                    continue
                s_, px, cur, ref = pool[int(rng.integers(len(pool)))]
                mode = str(rng.choice(["partial", "exact", "over", "none"]))
                vol = {"partial": max(1, cur // 2), "exact": cur, "over": cur + int(rng.integers(1, 50)),
                       "none": -int(rng.integers(0, 3))}[mode]
                typ = abi.MSG_CANCEL if rng.random() < 0.5 else abi.MSG_DELETE
                row.append((typ, s_, px, vol, int(kind == "cancel_ext"), ref))
            elif kind == "unknown":                        # an id that is not in the level: at an aggregate head, or no level at all
                if aggs and rng.random() < 0.6:
                    s_, px = aggs[int(rng.integers(len(aggs)))][:2]
                else:
                    s_, px = side, best + sgn * 37
                vol = 0 if rng.random() < 0.6 else int(rng.integers(1, 20))
                agent = rng.random() < 0.5
                row.append((abi.MSG_DELETE, s_, px, vol, int(not agent), UNKNOWN_ID if agent else (1 << 30) + 7))
            elif kind == "bad":
                row.append((int(rng.choice([abi.MSG_LIMIT, abi.MSG_MARKET])), side, best, -int(rng.integers(0, 3)), int(rng.integers(2)), 0))
            elif kind == "skip":
                t, d = (int(rng.choice([0, 5, 7, -1])), side) if rng.random() < 0.5 else (abi.MSG_LIMIT, int(rng.choice([2, -1])))
                row.append((t, d, best, 10, 0, 0))
            elif kind == "sweep":                          # more than the whole opposite side: the market order meets an empty side
                row.append((abi.MSG_MARKET, side, 0, 10**8, 1, 0))
        return row

    def oracle_submit(self, env, row, count, omap):
        o = self.oracles[env]
        o.clear_fills()
        refs = []
        for t, d, p, v, x, r in row[:count]:
            if not (1 <= t <= 4 and d in (0, 1)):
                refs.append(0)
                self.stats["skipped"] += 1
                continue
            if not x and t in (abi.MSG_CANCEL, abi.MSG_DELETE):
                r = omap.get(r, UNKNOWN_ID)
            refs.append(o.process_order(t, d, p, v, x, r))
        return np.array(refs, np.uint32), o.fills()

    def submit(self, rows, K, count=None, max_fills=4096, check=True, what="", orders=None):
        """rows -> submit_orders on the device (``orders``: the same rows as a device tensor, used instead of packing them here)
        and process_order on the oracles; then every output and book is compared."""
        import torch

        cnt = np.array([len(r) for r in rows] if count is None else count, np.int32)
        maps = [self.id_map(e) for e in range(self.n)]
        err0 = self.sim.errors()
        orders = pack(rows, K) if orders is None else orders
        refs, fills, n_fills = self.sim.submit_orders(orders, torch.tensor(cnt, device="cuda"), max_fills=max_fills)
        refs, nf = u32(refs), n_fills.cpu().numpy()
        clamp = np.clip(cnt, 0, K)
        st = self.sim.state()
        for e in range(self.n):
            orefs, ofills = self.oracle_submit(e, rows[e], int(clamp[e]), maps[e])
            if not check:
                continue
            assert not refs[e, clamp[e]:].any(), (what, e)
            if self.excluded[e] or H.capacity_excluded(st["err"][e], self.oracles[e], self.cfg, (what, e)):
                self.excluded[e] = True
                continue
            r = refs[e, : clamp[e]]
            assert np.array_equal(r == 0, orefs == 0) and np.array_equal(r == 0xFFFFFFFF, orefs == 0xFFFFFFFF), (what, e, r, orefs)
            got = fills_of(fills, nf, e)
            assert nf[e] == len(ofills) and H.canon_fills(got) == H.canon_fills(ofills), (what, e, nf[e], len(ofills))
            self.compare(e, (what, e))
            self.stats["rested"] += int(np.count_nonzero(r))
            self.stats["fills"] += int(nf[e])
            new = int(st["err"][e]) & ~int(err0[e])
            self.stats["bad_volume"] += bool(new & abi.ERR_BAD_VOLUME)
            self.stats["empty_book"] += bool(new & abi.ERR_EMPTY_BOOK)
        return refs, fills, nf

    def compare(self, e, what):
        from test_gpu_parity import compare_books

        st, os_ = self.sim.state(), self.oracles[e].state()
        for f in FIELDS:
            assert np.array_equal(st[f][e], os_[f]), (what, f, st[f][e], os_[f])
        assert H.close(st["cash"][e], os_["cash"]) and H.close(st["price"][e], os_["price"]), what
        compare_books(self.sim, e, self.oracles[e], what)

    def compare_all(self, what):
        st = self.sim.state()
        for e in range(self.n):
            if self.excluded[e] or H.capacity_excluded(st["err"][e], self.oracles[e], self.cfg, (what, e)):
                self.excluded[e] = True
                continue
            self.compare(e, (what, e))


STARTS = [10 * (3 + 7 * i) for i in range(24)]


def test_parity_with_oracle(kernel_family):
    """Five rounds of random programs (K = 40, ragged counts) on 24 books, with replays in between, against the oracle."""
    rng = np.random.default_rng(7)
    bed = Bed(STARTS)
    bed.replay(5)
    K = 40
    for rnd in range(5):
        rows = [bed.program(rng, e, K, None if rnd < 4 or e % 8 else ["rest", "mkt", "sweep"]) for e in range(bed.n)]
        bed.submit(rows, K, what=f"round {rnd}")
        bed.replay(int(rng.choice([1, 7, 20])))
        bed.compare_all(f"replay after round {rnd}")
    s = bed.stats
    assert s["rested"] > 50 and s["fills"] > 50 and s["bad_volume"] > 0 and s["empty_book"] > 0 and s["skipped"] > 0, s
    assert (~bed.excluded).sum() >= bed.n // 2, "most envs stay in the comparison"
    bed.sim.close()


def test_bit_identical_to_process_orders(kernel_family):
    """Twin handles on the same programs: one through submit_orders (and against the oracle), one through process_orders with
    the rows concatenated env by env.  Agent ids, refs, fills, books and state are all equal (the flat-form bit aside:
    process_orders converts every blob to the sorted form first)."""
    from test_gpu_parity import make_sim

    rng = np.random.default_rng(11)
    s = _stream(seed=43)
    bed = Bed(STARTS, s)
    b = make_sim(abi.default_cfg(n_envs=bed.n, **KW), [s])
    b.reset_book(0, np.array(STARTS, np.int32))
    bed.replay(5)
    b.replay(5)
    K = 32
    kinds = ["rest"] * 5 + ["cross"] * 2 + ["ext_limit"] * 2 + ["mkt", "ext_mkt"] + ["cancel_agent"] * 4 + ["cancel_ext", "unknown", "bad"]
    a = bed.sim
    for rnd in range(4):
        rows = [bed.program(rng, e, K, kinds) for e in range(bed.n)]
        refs, fills, nf = bed.submit(rows, K, what=f"twin {rnd}")
        flat = np.array([(e,) + o[:5] + (o[5] & 0xFFFFFFFF, 0) for e, row in enumerate(rows) for o in row], abi.ORDER_DTYPE)
        bfills, brefs = b.process_orders(flat, max_fills=1 << 16)
        assert np.array_equal(np.concatenate([refs[e, : len(r)] for e, r in enumerate(rows)]), brefs), rnd
        afills = np.concatenate([fills_of(fills, nf, e) for e in range(bed.n)])
        assert afills.tobytes() == bfills.tobytes(), rnd
        sa, sb = a.state(), b.state()
        for f in abi.ENV_STATE_DTYPE.names:
            x, y = sa[f], sb[f]
            if f == "reserved":
                x, y = x & np.uint32(0xFFFFFFFE), y & np.uint32(0xFFFFFFFE)
            assert np.array_equal(x, y, equal_nan=True), (rnd, f)
        for e in range(bed.n):
            for side in (0, 1):
                assert np.array_equal(a.dump_book(e, side), b.dump_book(e, side)), (rnd, e, side)
                assert np.array_equal(a.dump_agent_orders(e, side), b.dump_agent_orders(e, side)), (rnd, e, side)
        bed.replay(3)
        b.replay(3)
    b.close()
    a.close()


def test_count_zero_dead_envs_and_clamping(kernel_family):
    """Rows with count 0 (and counts below 0) leave their env exactly as it was, whatever the row holds; a dead env ignores its
    orders; a count above K is K."""
    import torch

    bed = Bed(STARTS[:9])
    bed.replay(5)
    K = 6
    # env 0 dies: an external market sell larger than the whole buy side
    bed.submit([[(abi.MSG_MARKET, 1, 0, 10**8, 1, 0)]] + [[]] * 8, K)
    assert bed.sim.state()["err"][0] & abi.ERR_EMPTY_BOOK
    before = bed.sim.state()
    books = [[bed.sim.dump_book(e, s) for s in (0, 1)] for e in range(bed.n)]
    rows = [[(abi.MSG_LIMIT, 0, int(o.state()["best_buy"]) - 200, 10, 0, 0)] * K for o in bed.oracles]   # all rest
    count = np.array([2, 0, -4, 0, 3, 0, 100, 0, 0], np.int32)
    refs, fills, nf = bed.submit(rows, K, count=count)
    after = bed.sim.state()
    for e in (0, 1, 2, 3, 5, 7, 8):
        assert after[e].tobytes() == before[e].tobytes(), e
        assert all(np.array_equal(bed.sim.dump_book(e, s), books[e][s]) for s in (0, 1)), e
        assert not refs[e].any() and nf[e] == 0, e
    assert np.count_nonzero(refs[4]) == 3 and np.count_nonzero(refs[6]) == K      # count 3, and 100 clamped to K = 6
    assert torch.equal(bed.sim.submit_orders(pack(rows, K), 0)[2], torch.zeros(bed.n, dtype=torch.int32, device="cuda"))
    bed.sim.close()


def test_portfolio_and_fill_log_unchanged(kernel_family):
    """After env steps the agent has inventory, cash and a fill log; a submission that fills the agent's orders and trades
    through its own market orders changes none of them (Exchange.process_order returns its fills)."""
    import torch

    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(episode_steps=400, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7, fill_log_capacity=256)
    bed = Bed(STARTS[:7], env=True, **kw)
    rng = np.random.default_rng(3)
    ad = abi.action_dim(bed.cfg)
    for _ in range(6):
        a = rng.uniform(0.5, 6.0, size=(bed.n, ad))
        bed.sim.step(torch.tensor(a, device="cuda"))
        for e, o in enumerate(bed.oracles):
            o.step(a[e])
    st0 = bed.sim.state()
    logs = [bed.sim.fills(e) for e in range(bed.n)]
    assert any(len(x) for x in logs) and np.any(st0["inventory"] != 0)
    rows = []
    for e in range(bed.n):
        st = bed.oracles[e].state()
        rows.append([(abi.MSG_MARKET, 0, 0, 150, 1, 0), (abi.MSG_MARKET, 1, 0, 150, 1, 0), (abi.MSG_MARKET, 0, 0, 40, 0, 0),
                     (abi.MSG_LIMIT, 1, int(st["best_buy"]), 30, 0, 0)])
    _, _, nf = bed.submit(rows, 4, what="fills the agent")
    assert nf.sum() > 0
    st1 = bed.sim.state()
    assert np.array_equal(st1["inventory"], st0["inventory"]) and np.array_equal(st1["cash"], st0["cash"])
    assert np.array_equal(st1["price"], st0["price"], equal_nan=True)
    for e in range(bed.n):
        assert bed.sim.fills(e).tobytes() == logs[e].tobytes(), e
    bed.sim.close()


def test_max_fills_truncation(kernel_family):
    """max_fills = 3: n_fills is the whole count, the first three fills are written, FILL_LOG_FULL exactly where n_fills > 3."""
    from test_gpu_parity import make_sim

    s = _stream(seed=47)
    a, b = make_sim(abi.default_cfg(n_envs=8, **KW), [s]), make_sim(abi.default_cfg(n_envs=8, **KW), [s])
    starts = np.array(STARTS[:8], np.int32)
    for h in (a, b):
        h.reset_book(0, starts)
        h.replay(4)
    rows = [[(abi.MSG_MARKET, e % 2, 0, 40 * e + 1, 1, 0), (abi.MSG_MARKET, 1 - e % 2, 0, 60 * e + 1, 0, 0)] for e in range(8)]
    _, fa, na = a.submit_orders(pack(rows, 2), max_fills=3)
    _, fb, nb = b.submit_orders(pack(rows, 2), max_fills=512)
    na, nb = na.cpu().numpy(), nb.cpu().numpy()
    assert np.array_equal(na, nb) and na.max() > 3 and na.min() <= 3
    full = a.errors() & abi.ERR_FILL_LOG_FULL
    assert np.array_equal(full != 0, na > 3)
    assert not (b.errors() & abi.ERR_FILL_LOG_FULL).any()
    for e in range(8):
        assert fills_of(fa, na, e).tobytes() == fills_of(fb, nb, e)[:3].tobytes(), e
    a.close()
    b.close()


def test_capacity_flags(kernel_family):
    """64 levels / 256 orders / 32 agent orders per side: 70 external limits at new prices (LEVEL_OVERFLOW), 40 agent limits
    (AGENT_OVERFLOW), 300 external limits at one price (ORDER_OVERFLOW) -- the error bits are the oracle's high-water marks."""
    kw = dict(max_agent_orders=32)
    bed = Bed(STARTS[:4], **kw)
    bed.replay(3)
    K = 300
    rows = []
    for e in range(4):
        st = bed.oracles[e].state()
        bb = int(st["best_buy"])
        if e == 0:
            rows.append([(abi.MSG_LIMIT, 0, bb - 100 * k - 50, 5, 1, (1 << 29) + k) for k in range(70)])
        elif e == 1:
            rows.append([(abi.MSG_LIMIT, 0, bb - 100 * (k % 5), 5, 0, 0) for k in range(40)])
        elif e == 2:
            rows.append([(abi.MSG_LIMIT, 0, bb - 300, 1, 1, (1 << 29) + k) for k in range(300)])
        else:
            rows.append([(abi.MSG_LIMIT, 1, int(st["best_sell"]), 5, 0, 0)] * 10)
    bed.submit(rows, K, check=False)
    err = bed.sim.errors()
    for e, bit in enumerate((abi.ERR_LEVEL_OVERFLOW, abi.ERR_AGENT_OVERFLOW, abi.ERR_ORDER_OVERFLOW, 0)):
        o = bed.oracles[e]
        want = H.exceeded_bits(o.peaks(), bed.cfg) | int(o.state()["err"])
        assert int(err[e]) == want, (e, int(err[e]), want, o.peaks())
        assert want & bit == bit
    bed.compare(3, "no capacity exceeded")
    bed.sim.close()


def test_flat_blobs_submit_then_replay(kernel_family):
    """k_replay_flat leaves thin books flat; orders submitted to half of them (count 0 elsewhere, rows built from the oracle so
    that no host dump converts the blobs first) match the oracle, the other books stay flat, and the replay after it is the
    tracked kernel (no flat blob afterwards) and follows the oracle."""
    import torch

    shape = "thin"
    s = A.build(shape, A.SHAPES[shape]["seeds"][0])
    starts = [10 * t for t in A.STARTS]
    cfg_kw = {k: getattr(A.cfg_for(shape, n_envs=1, resync=0, outer_levels=2), k)
              for k in ("n_levels", "max_levels_per_side", "max_orders_per_side", "max_agent_orders", "resync", "outer_levels", "step_us")}
    bed = Bed(starts, s, **cfg_kw)
    done, flat = 0, np.zeros(bed.n, bool)
    while done < 120 and not flat.any():
        bed.replay(7)
        done += 7
        flat = (bed.sim.state()["reserved"] & 1) != 0
    if kernel_family == "fast":
        assert flat.any(), "some books are flat"
    rng = np.random.default_rng(5)
    K = 12
    rows = []
    for e, o in enumerate(bed.oracles):
        st = o.state()
        bb, bs = int(st["best_buy"]), int(st["best_sell"])
        row = []
        if e % 2 == 0 and bb and bs != INT_MAX:
            for _ in range(K):
                side = int(rng.integers(2))
                best, other, sgn = (bb, bs, -1) if side == 0 else (bs, bb, 1)
                r = rng.random()
                if r < 0.6:
                    row.append((abi.MSG_LIMIT, side, best + sgn * 100 * int(rng.integers(0, 4)), int(rng.integers(1, 30)), 0, 0))
                elif r < 0.8:
                    row.append((abi.MSG_LIMIT, side, other, int(rng.integers(1, 30)), 0, 0))
                else:
                    row.append((abi.MSG_MARKET, side, 0, int(rng.integers(1, 30)), int(rng.integers(2)), 0))
        rows.append(row)
    cnt = np.array([len(r) for r in rows], np.int32)
    refs, fills, nf = bed.sim.submit_orders(pack(rows, K), torch.tensor(cnt, device="cuda"), max_fills=4096)
    now_flat = (bed.sim.state()["reserved"] & 1) != 0
    assert np.array_equal(now_flat, flat & (cnt == 0)), (flat, now_flat, cnt)
    refs, nf = u32(refs), nf.cpu().numpy()
    for e, o in enumerate(bed.oracles):
        orefs, ofills = bed.oracle_submit(e, rows[e], len(rows[e]), {})
        assert np.array_equal(refs[e, : len(rows[e])] == 0, orefs == 0), e
        assert H.canon_fills(fills_of(fills, nf, e)) == H.canon_fills(ofills), e
    assert int(np.concatenate(bed.sim.state()["n_agent_orders"]).sum()) > 0
    for k in (1, 10, 23):            # (no host dump before the first replay: it would convert the flat blobs itself)
        bed.replay(k)
        assert not (bed.sim.state()["reserved"] & 1).any(), "the tracked replay leaves no flat blob"
        bed.compare_all(f"replay {k} after submit")
    bed.sim.close()


def test_env_steps_and_rollouts_after_submit(kernel_family):
    """Agent orders submitted inside and far outside the quote ladder, then env steps and a fused rollout: the Beta-ladder diff
    sees them (the far ones are the wide cancels) -- obs, rewards and books == the oracle."""
    import torch

    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(episode_steps=400, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7)
    bed = Bed(STARTS[:10], env=True, **kw)
    rng = np.random.default_rng(9)
    ad = abi.action_dim(bed.cfg)
    K = 16
    for rnd in range(3):
        rows = []
        for e in range(bed.n):
            st = bed.oracles[e].state()
            bb, bs = int(st["best_buy"]), int(st["best_sell"])
            row = [(abi.MSG_LIMIT, 0, bb - 100 * int(k), int(rng.integers(1, 50)), 0, 0) for k in rng.integers(0, 12, size=4)]
            row += [(abi.MSG_LIMIT, 1, bs + 100 * int(k), int(rng.integers(1, 50)), 0, 0) for k in rng.integers(0, 12, size=4)]
            row += bed.program(rng, e, 6, ["cancel_agent", "rest", "cross"])
            rows.append(row)
        bed.submit(rows, K, what=f"round {rnd}")
        for t in range(3):
            a = rng.uniform(0.5, 6.0, size=(bed.n, ad))
            obs, rew, done = (x.cpu().numpy() for x in bed.sim.step(torch.tensor(a, device="cuda")))
            for e, o in enumerate(bed.oracles):
                oo, orw, od = o.step(a[e])
                if not bed.excluded[e]:
                    H.assert_close_vec(obs[e], oo, (rnd, t, e))
                    assert H.close(rew[e], orw) and bool(done[e]) == od, (rnd, t, e)
            bed.compare_all((rnd, "step", t))
        agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 0))
        obs, act, rew, done = (x.cpu().numpy() for x in bed.sim.rollout(3, agent))
        for e, o in enumerate(bed.oracles):
            oo, oa, orw, od = o.rollout(3, agent)
            if not bed.excluded[e]:
                for t in range(3):
                    H.assert_close_vec(obs[t, e], oo[t], (rnd, "rollout", t, e))
                    assert H.close(rew[t, e], orw[t]), (rnd, t, e)
        bed.compare_all((rnd, "rollout"))
    bed.sim.close()


def _requote(count, price, ids, best, tick=100):
    """On the device, from agent_orders() and book_depth(): a DELETE with volume None of every resting agent order (by id),
    then one limit per side at the best price and one a tick behind it, 5 shares each.  Unused slots are type 0 (skipped)."""
    import torch

    N, _, A_ = price.shape
    dev = price.device
    live = torch.arange(A_, device=dev)[None, None, :] < count[:, :, None]
    cancel_type = torch.where(live, abi.MSG_DELETE, 0).reshape(N, 2 * A_)
    cancel_side = torch.arange(2, device=dev)[None, :, None].expand(N, 2, A_).reshape(N, 2 * A_)
    b = best.to(torch.int64)
    quote_price = torch.stack([b[:, 0], b[:, 0] - tick, b[:, 1], b[:, 1] + tick], dim=1)
    typ = torch.cat([cancel_type, torch.full((N, 4), abi.MSG_LIMIT, device=dev)], dim=1)
    side = torch.cat([cancel_side, torch.tensor([0, 0, 1, 1], device=dev).expand(N, 4)], dim=1)
    px = torch.cat([price.reshape(N, 2 * A_).to(torch.int64), quote_price], dim=1)
    vol = torch.cat([torch.zeros((N, 2 * A_), dtype=torch.int64, device=dev), torch.full((N, 4), 5, device=dev)], dim=1)
    ref = torch.cat([ids.reshape(N, 2 * A_).to(torch.int64), torch.zeros((N, 4), dtype=torch.int64, device=dev)], dim=1)
    return abi.pack_orders(typ, side, px, vol, 0, ref)


def test_agent_orders_requote_forward_step_loop(kernel_family):
    """The simulator-level loop on the device: agent_orders() -> cancel every order by id and re-quote at the touch with
    submit_orders -> forward_step, several rounds, against the oracle (fed the same orders from the host)."""
    bed = Bed(STARTS[:12])
    bed.replay(5)
    A_ = 16
    for rnd in range(6):
        count, price, _, ids = bed.sim.agent_orders(A_, queue=False)
        orders = _requote(count, price, ids, bed.sim.book_depth(1)[0][:, :, 0])
        K = orders.shape[1]
        host = orders.cpu().numpy().view(abi.ORDER_DTYPE).reshape(bed.n, K)
        rows = [[tuple(int(x[f]) for f in ("type", "direction", "price", "volume", "is_external", "ref")) for x in host[e]]
                for e in range(bed.n)]
        cnt = count.cpu().numpy()
        for e in range(bed.n):
            assert sum(r[0] == abi.MSG_DELETE for r in rows[e]) == min(A_, cnt[e, 0]) + min(A_, cnt[e, 1])
        bed.submit(rows, K, what=f"requote {rnd}", orders=orders)
        bed.forward_step(int(np.random.default_rng(rnd).choice([3, 10, 20])))
        bed.compare_all(f"forward_step {rnd}")
    assert int(bed.sim.agent_orders(A_, queue=False)[0].sum()) > 0
    bed.sim.close()


def test_cuda_graph_capture(kernel_family):
    """submit_orders(out=...) + forward_step captured once in a CUDA graph on a side stream and replayed: == an eager twin."""
    import torch

    from test_gpu_parity import make_sim

    s = _stream(seed=53)
    n = 12
    g, e_ = make_sim(abi.default_cfg(n_envs=n, **KW), [s]), make_sim(abi.default_cfg(n_envs=n, **KW), [s])
    for h in (g, e_):
        h.reset_book(0, np.array(STARTS[:n], np.int32))
        h.replay(5)
    st = g.state()
    bb, bs = torch.tensor(st["best_buy"].astype(np.int64)), torch.tensor(st["best_sell"].astype(np.int64))
    typ = torch.tensor([abi.MSG_LIMIT, abi.MSG_LIMIT, abi.MSG_MARKET, abi.MSG_DELETE])[None, :].expand(n, 4)
    side = torch.tensor([0, 1, 0, 0])[None, :].expand(n, 4)
    price = torch.stack([bb, bs, bb, bb - 100], dim=1)
    orders = abi.pack_orders(typ, side, price, torch.tensor([7, 9, 3, 0])[None, :].expand(n, 4), 0, 1).cuda()
    count = torch.tensor([4, 0, 3, 4, 2, 4, 1, 4, 4, 3, 4, 4], dtype=torch.int32, device="cuda")
    out = (torch.empty((n, 4), dtype=torch.uint32, device="cuda"), torch.empty((n, 8, 6), dtype=torch.int32, device="cuda"),
           torch.empty(n, dtype=torch.int32, device="cuda"))
    side_stream = torch.cuda.Stream()
    side_stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side_stream):
        g.submit_orders(orders, count, max_fills=8, out=out, stream=side_stream)
        g.forward_step(2, stream=side_stream)
    torch.cuda.current_stream().wait_stream(side_stream)
    e_.submit_orders(orders, count, max_fills=8)
    e_.forward_step(2)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g.submit_orders(orders, count, max_fills=8, out=out)
        g.forward_step(2)
    for k in range(5):
        graph.replay()
        r, f, nf = e_.submit_orders(orders, count, max_fills=8)
        e_.forward_step(2)
        torch.cuda.synchronize()
        assert torch.equal(out[0].view(torch.int32), r.view(torch.int32)) and torch.equal(out[2], nf), k
        for env in range(n):
            m = min(int(nf[env]), 8)
            assert torch.equal(out[1][env, :m], f[env, :m]), (k, env)
        assert torch.equal(g.state_dev(), e_.state_dev()), k
    assert int(out[2].sum()) > 0 and int((out[0].view(torch.int32) != 0).sum()) > 0
    for env in range(n):
        for sd in (0, 1):
            assert np.array_equal(g.dump_book(env, sd), e_.dump_book(env, sd)), (env, sd)
    g.close()
    e_.close()


@pytest.mark.fast_only        # deep-book capacities always run the general kernel on the blobs in HBM
def test_deep_book_mode():
    """256 levels x 16 384 orders per side (blobs worked on in place in HBM) against the unbounded oracle."""
    sc = dict(n_msgs=200_000, duration_s=400, n_levels=50, mid0=2_000_000, p_limit=0.40, p_cancel=0.15, p_delete=0.37, p_exec=0.08,
              geom_p=0.10, init_levels=70, mean_queue=80, target_orders=6000, max_offset_ticks=80, p_sweep=0.0)
    s = _stream(seed=11, **sc)
    bed = Bed([100, 1500, 3000], s, n_levels=50, outer_levels=20, max_levels_per_side=256, max_orders_per_side=16384)
    assert bed.sim.kernel_path == "deep"
    bed.replay(5)
    rng = np.random.default_rng(13)
    for rnd in range(3):
        bed.submit([bed.program(rng, e, 48) for e in range(bed.n)], 48, what=f"deep {rnd}")
        bed.replay(7)
        bed.compare_all(f"deep replay {rnd}")
    assert bed.stats["rested"] > 0 and bed.stats["fills"] > 0
    bed.sim.close()


def test_arguments(kernel_family):
    """NULL or out-of-range arguments are LOBSIM_E_INVALID without a launch; the façade checks its tensors and out=; a valid call
    is exactly one launch."""
    import torch

    from rl4mm_b200._lib import LobsimError, lib

    sim = Bed(STARTS[:3]).sim
    orders = pack([[(abi.MSG_LIMIT, 0, 1_000_000, 5, 0, 0)]] * 3, 4)
    count = torch.ones(3, dtype=torch.int32, device="cuda")
    r, f, nf = sim.submit_orders(orders, count, max_fills=4)
    L = lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    good = [4, P(orders), P(count), P(r), 4, P(f), P(nf)]
    c = sim.launch_count
    assert L.lobsim_submit_orders_dev(sim._h, *good, st) == abi.OK and sim.launch_count == c + 1
    bad = [(0, 0), (0, -1), (1, None), (2, None), (4, -1), (5, None)]
    mis = ctypes.c_void_p(orders.data_ptr() + 4)
    for i, v in bad + [(1, mis)]:
        args = list(good)
        args[i] = v
        c = sim.launch_count
        assert L.lobsim_submit_orders_dev(sim._h, *args, st) == abi.E_INVALID, (i, v)
        assert sim.launch_count == c
    assert L.lobsim_submit_orders_dev(None, *good, st) == abi.E_INVALID
    assert L.lobsim_submit_orders_dev(sim._h, 4, P(orders), P(count), None, 0, None, None, st) == abi.OK   # outputs optional
    for bad_orders in (orders.to(torch.int64), orders[:2], orders.cpu(), orders[:, :, :7], orders.transpose(0, 1)):
        with pytest.raises(ValueError):
            sim.submit_orders(bad_orders)
    with pytest.raises(ValueError):
        sim.submit_orders(orders, count.to(torch.int64))
    with pytest.raises(ValueError):
        sim.submit_orders(orders, max_fills=-1)
    with pytest.raises(ValueError):
        sim.submit_orders(orders, max_fills=4, out=(r, f))
    with pytest.raises(ValueError):
        sim.submit_orders(orders, max_fills=5, out=(r, f, nf))
    with pytest.raises(ValueError):
        sim.submit_orders(orders, max_fills=4, refs=False, out=(r, f, nf))
    assert sim.submit_orders(orders, max_fills=4, refs=False, out=(None, f, nf))[0] is None
    with pytest.raises(ValueError):
        sim.submit_orders(orders[:, :0].contiguous())                      # K = 0
    with pytest.raises(LobsimError):
        sim.book_depth(0)                                                  # (the façade's errors are LobsimError / ValueError)
    sim.close()
