"""Seeded random programs over the whole C ABI against one oracle per env.  Every other test drives one call family in one fixed
order; the handle carries state from call to call (books left in the flat form, the replay fast path gated by "an agent order may
rest", the fill log of the last call, per-env streams), so a wrong transition only shows up on some orders of calls.  A program is
about 30 calls drawn from reset / reset_book (all envs or a subset), replay, replay_host, forward_step, process_orders, set_book,
step, step_host, rollout, rollout_info and rollout_agents, on one handle of 2-40 envs with 1-3 message streams, capacities of a
compiled layout or a general triple, and a fill log on or off.  After every call: state() field by field, the L3 and agent books
and the fills of the call against the oracle; state(), state_dev() and errors() agree; episode_stats_dev == episode_stats.
Soak runs: LOBSIM_SEQ_CASES=500 LOBSIM_SEQ_SEED0=... pytest tests/test_gpu_call_sequences.py"""
import ctypes
import os

import numpy as np
import pytest

import parity_helpers as H
from rl4mm_b200 import abi, synthetic

pytestmark = pytest.mark.gpu

N_CASES = int(os.environ.get("LOBSIM_SEQ_CASES", "12"))
SEED0 = int(os.environ.get("LOBSIM_SEQ_SEED0", "0"))
DEATH_BITS = abi.ERR_EMPTY_BOOK | abi.ERR_NO_SNAPSHOT | abi.ERR_END_OF_STREAM | abi.ERR_BAD_ACTION
CAPS = [(64, 256, 32), (128, 512, 64), (64, 256, 64), (128, 256, 64), (96, 384, 48)]   # the last one has no compiled layout
FIELDS = ("inventory", "now_step", "episode_start_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume",
          "best_sell_volume", "err", "n_agent_orders")
DURATION_S = 200


def _streams(rng, n):
    out = []
    for i in range(n):
        sc = synthetic.SynthConfig(seed=int(rng.integers(1 << 30)), n_msgs=60_000, duration_s=DURATION_S, n_levels=10,
                                   mid0=int(rng.choice([500_000, 2_000_000])), p_limit=0.45, p_cancel=0.15, p_delete=0.3, p_exec=0.1,
                                   geom_p=float(rng.choice([0.2, 0.35])), init_levels=12, mean_queue=int(rng.choice([2, 4])),
                                   target_orders=int(rng.choice([25, 60, 150])), max_offset_ticks=int(rng.choice([12, 30])),
                                   p_sweep=float(rng.choice([0.005, 0.03])))
        out.append(synthetic.generate(sc))
    return out


def _cfg_kw(rng):
    nl, no, na = CAPS[int(rng.integers(len(CAPS)))]
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6),
             abi.feature(abi.FEAT_PRICE_MOVE, 3, 100_000, -1e4, 1e4), abi.feature(abi.FEAT_TRADE_DIR_IMBALANCE, 5, 100_000, -1, 1)]
    return dict(n_levels=10, episode_steps=int(rng.choice([15, 10_000])), warmup_steps=10, outer_levels=int(rng.choice([5, 9])),
                resync=1, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
                terminal_reward=abi.Reward(abi.REWARD_INV_ADJ_PNL, 0, 0.1), initial_cash=1e8, portfolio_carryover=0,
                max_levels_per_side=nl, max_orders_per_side=no, max_agent_orders=na, fill_log_capacity=int(rng.choice([0, 4096])))


def _agent(rng, kind=None):
    kind = kind or str(rng.choice(["none", "fixed", "random", "teradactyl", "external"]))
    if kind == "fixed":
        return abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(*rng.uniform(0.5, 6, 4), 0.0))
    if kind == "random":
        return abi.Agent(kind=abi.AGENT_RANDOM, fixed_action=(ctypes.c_double * 5)(6.0, 6.0, 6.0, 6.0, 0.0),
                         reserved=int(rng.integers(1 << 20)))
    if kind == "teradactyl":
        return abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=1, max_inventory=float(rng.choice([50.0, 500.0])),
                         default_kappa=float(rng.uniform(3, 10)), default_omega=float(rng.uniform(0.2, 0.8)),
                         max_kappa=float(rng.uniform(10, 14)), exponent=float(rng.choice([1.0, 2.0])))
    return abi.Agent(kind=abi.AGENT_EXTERNAL if kind == "external" else abi.AGENT_NONE)


def _random_book(rng, mid, caps, ref0):
    """A valid L3 book (dump_book format): optional snapshot aggregate at the head of a level, external orders, agent orders whose
    ids increase along every FIFO with room for the external orders queued between them."""
    sides, next_id = [], 1
    for side in (0, 1):
        ents = []
        for k in range(int(rng.integers(1, 9))):
            px = mid - 100 * (k + 1) if side == 0 else mid + 100 * (k + 1)
            if rng.random() < 0.3:
                ents.append((px, int(rng.integers(1, 500)), abi.REF_AGGREGATE, k))
            for _ in range(int(rng.integers(0 if ents and ents[-1][0] == px else 1, 4))):
                if rng.random() < 0.4 and sum((e[2] & abi.REF_AGENT) != 0 for e in ents) < min(caps[2], 6):
                    next_id += 2
                    ents.append((px, int(rng.integers(1, 60)), abi.REF_AGENT | next_id, k))
                else:
                    ref0 += 1
                    next_id += 1
                    ents.append((px, int(rng.integers(1, 300)), ref0, k))
        sides.append(np.array(ents, abi.BOOK_ENTRY_DTYPE))
    return sides, ref0


class Program:
    def __init__(self, seed):
        from oracle.oracle import Oracle
        from test_gpu_parity import make_sim

        rng = self.rng = np.random.default_rng(20_000 + seed)
        self.seed = seed
        n = int(rng.integers(2, 41))
        while n % 4 == 0:                                   # never a whole number of CTAs
            n = int(rng.integers(2, 41))
        self.n = n
        self.streams = _streams(rng, int(rng.integers(1, 4)))
        self.kw = _cfg_kw(rng)
        self.cfg = abi.default_cfg(n_envs=n, **self.kw)
        self.sim = make_sim(self.cfg, self.streams)
        self.oracles = [Oracle(abi.default_cfg(**self.kw), self.streams[0], env_index=e) for e in range(n)]
        self.sid = np.zeros(n, np.int32)
        self.excluded = np.zeros(n, bool)        # capacity flagged or the reference raised: outputs not compared until a reset
        self.ref = 1 << 28                       # external refs of the orders this program makes up
        self.checked = 0

    # ---- calls -------------------------------------------------------------------------------------------------------------
    def _starts(self, ids, lo, hi):
        return (self.rng.integers(lo, hi, size=len(ids)) * 10).astype(np.int32)

    def reset(self, book_only, all_envs=False):
        rng, n = self.rng, self.n
        ids = np.arange(n) if all_envs or rng.random() < 0.5 else np.sort(rng.choice(n, size=int(rng.integers(1, n + 1)), replace=False))
        sids = rng.integers(0, len(self.streams), size=len(ids)).astype(np.int32)
        starts = self._starts(ids, 2, DURATION_S // 2)
        env_ids = None if len(ids) == n and rng.random() < 0.5 else ids
        if book_only:
            self.sim.reset_book(sids, starts, env_ids=env_ids)
        else:
            self.sim.reset(sids, starts, env_ids=env_ids)
            self.has_reset = True
        for i, e in enumerate(ids):
            o = self.oracles[e]
            self.sid[e] = sids[i]
            o.set_stream(self.streams[sids[i]])
            if book_only:
                o.reset_book(int(starts[i]))
            else:
                o.reset(int(starts[i]))
                self.excluded[e] = False
        return f"{'reset_book' if book_only else 'reset'} {len(ids)} envs"

    def replay(self, how):
        k = int(self.rng.choice([0, 1, 7, 10, 57]))
        if how == "forward_step":
            self.sim.forward_step(k)
            for o in self.oracles:
                o.forward_step(k)
        elif how == "replay_host":
            sid = int(self.rng.integers(len(self.streams)))
            s = self.streams[sid]
            now = self.sim.state()["now_step"][self.sid == sid]
            first, last = 0, 0
            if len(now):
                first = int(s.step_off[max(0, min(int(now.min()), s.n_grid_steps))])
                last = int(s.step_off[max(0, min(int(now.max()) + k, s.n_grid_steps))])
            st = np.zeros(self.n, abi.ENV_STATE_DTYPE)
            self.sim.replay_host(sid, s.msgs[first:max(first, last)].copy(), first, k, st)
            self.host_state = st
            for o in self.oracles:
                o.replay(k)
        else:
            self.sim.replay(k)
            for o in self.oracles:
                o.replay(k)
        return f"{how}({k})", "replay"

    def process_orders(self):
        rng = self.rng
        envs = np.sort(rng.choice(self.n, size=int(rng.integers(1, min(self.n, 6) + 1)), replace=False))
        dev, orc = [], []
        st = self.sim.state()
        for e in envs:
            o = self.oracles[e]
            bb, bs = int(st["best_buy"][e]), int(st["best_sell"][e])
            if bb == 0 or bs == 2**31 - 1:
                continue
            for _ in range(int(rng.integers(1, 5))):
                r = rng.random()
                side = int(rng.integers(2))
                if r < 0.45:            # agent limit inside or behind the book
                    px = (bb - 100 * int(rng.integers(-1, 4))) if side == 0 else (bs + 100 * int(rng.integers(-1, 4)))
                    vol = int(rng.integers(1, 80))
                    dev.append((e, abi.MSG_LIMIT, side, px, vol, 0, 0, 0)); orc.append((e, abi.MSG_LIMIT, side, px, vol, 0, 0))
                elif r < 0.7:           # cancel / delete one of the env's resting agent orders (k-th by id on both)
                    da, oa = self.sim.dump_agent_orders(e, side), o.dump_agent_orders(side)
                    if not len(oa) or len(da) != len(oa):
                        continue
                    j = int(rng.integers(len(oa)))
                    typ = abi.MSG_CANCEL if rng.random() < 0.5 else abi.MSG_DELETE
                    vol = int(rng.integers(1, int(oa[j]["volume"]) + 1)) if typ == abi.MSG_CANCEL else 0
                    dev.append((e, typ, side, int(da[j]["price"]), vol, 0, int(da[j]["ref"]) & 0x7fffffff, 0))
                    orc.append((e, typ, side, int(oa[j]["price"]), vol, 0, int(oa[j]["ref"]) & 0x7fffffff))
                elif r < 0.85:          # agent market order
                    vol = int(rng.integers(1, 150))
                    dev.append((e, abi.MSG_MARKET, side, 0, vol, 0, 0, 0)); orc.append((e, abi.MSG_MARKET, side, 0, vol, 0, 0))
                else:                   # an external limit order
                    self.ref += 1
                    px = (bb - 100 * int(rng.integers(0, 3))) if side == 0 else (bs + 100 * int(rng.integers(0, 3)))
                    vol = int(rng.integers(1, 200))
                    dev.append((e, abi.MSG_LIMIT, side, px, vol, 1, self.ref, 0)); orc.append((e, abi.MSG_LIMIT, side, px, vol, 1, self.ref))
        fills, refs = self.sim.process_orders(np.array(dev, abi.ORDER_DTYPE))
        ofills, orefs = [], []
        for e, typ, side, px, vol, ext, ref in orc:
            o = self.oracles[e]
            o.clear_fills()
            orefs.append(o.process_order(typ, side, px, vol, ext, ref))
            ofills.append(o.fills())
        involved = np.array([d[0] for d in dev], int)
        if not (self.excluded[involved].any() or (self.sim.errors()[involved] & H.CAPACITY_BITS).any()):
            assert H.canon_fills(fills) == H.canon_fills(np.concatenate(ofills) if ofills else np.zeros(0, abi.FILL_DTYPE)), self.what
            assert np.array_equal(refs == 0, np.array(orefs) == 0) and np.array_equal(refs == 0xffffffff, np.array(orefs) == 0xffffffff), self.what
        return f"process_orders({len(dev)})"

    def set_book(self):
        rng = self.rng
        dst = int(rng.integers(self.n))
        src = int(rng.integers(self.n))
        o = self.oracles[dst]
        # another env's book: only from the same stream at the same or an earlier clock, so that no order of the copied book has
        # an external id that the stream hands out again later (two resting orders with one external id are undefined)
        copyable = src != dst and not self.excluded[src] and self.sid[src] == self.sid[dst] and \
            self.oracles[src].state()["now_step"] <= o.state()["now_step"]
        if rng.random() < 0.5 and copyable:
            self.sim.set_book(dst, self.sim.dump_book(src, 0), self.sim.dump_book(src, 1))
            o.set_book(self.oracles[src].dump_book(0), self.oracles[src].dump_book(1))
            what = f"set_book({dst} <- env {src})"
        else:
            st = o.state()
            mid = (int(st["best_buy"]) + int(st["best_sell"])) // 200 * 100 if st["best_buy"] and st["best_sell"] < 2**31 - 1 else 1_000_000
            (buy, sell), self.ref = _random_book(rng, mid, (self.cfg.max_levels_per_side, self.cfg.max_orders_per_side,
                                                            self.cfg.max_agent_orders), self.ref)
            self.sim.set_book(dst, buy, sell)
            o.set_book(buy, sell)
            what = f"set_book({dst} random)"
        assert self.sim.state()["err"][dst] == 0, what     # set_book clears the error bits
        return what

    def step(self, host):
        if not self.has_reset:
            return self.reset(False)
        a = self.rng.uniform(0.2, 6.0, size=(self.n, abi.action_dim(self.cfg)))
        if host:
            obs, rew, done = np.zeros((self.n, abi.obs_dim(self.cfg))), np.zeros(self.n), np.zeros(self.n, np.uint8)
            self.sim.step_host(a, obs, rew, done)
        else:
            import torch

            obs, rew, done = (x.cpu().numpy() for x in self.sim.step(torch.tensor(a, device="cuda")))
        flagged = self.sim.errors() & H.CAPACITY_BITS      # (justified or not: check() decides before it excludes the env)
        for e, o in enumerate(self.oracles):
            oo, orw, od = o.step(a[e])
            if self.excluded[e] or flagged[e] or o.state()["err"] & DEATH_BITS:
                continue
            H.assert_close_vec(obs[e], oo, f"{self.what} env {e} obs")
            assert H.close(rew[e], orw) and bool(done[e]) == od, (self.what, e)
        self.last_rew, self.last_done = rew[None], done[None]
        return f"step{'_host' if host else ''}"

    def rollout(self, how):
        import torch

        if not self.has_reset:
            return self.reset(False)
        T = int(self.rng.choice([1, 3, 12]))
        ad = abi.action_dim(self.cfg)
        if how == "agents":
            agents = [_agent(self.rng, str(self.rng.choice(["fixed", "random", "teradactyl"]))) for _ in range(self.n)]
            obs, act, rew, done, info = (x.cpu().numpy() for x in self.sim.rollout(T, agents, want_info=True))
        else:
            agent = _agent(self.rng)
            ext = torch.tensor(self.rng.uniform(0.2, 6.0, size=(T, self.n, ad)), device="cuda") if agent.kind == abi.AGENT_EXTERNAL else None
            out = [x.cpu().numpy() if x is not None else None for x in self.sim.rollout(T, agent, ext, want_info=how == "info")]
            obs, act, rew, done = out[:4]
            info = out[4] if how == "info" else None
            agents = [agent] * self.n
        flagged = self.sim.errors() & H.CAPACITY_BITS
        for e, o in enumerate(self.oracles):
            a = agents[e]
            oo, oa, orw, od, oi = o.rollout(T, a, act[:, e] if a.kind == abi.AGENT_EXTERNAL else None, want_info=True)
            if self.excluded[e] or flagged[e]:
                continue
            for t in range(T):
                if int(oi[t, abi.INFO_FIELDS.index("err")]) & (DEATH_BITS | H.CAPACITY_BITS):
                    break
                w = f"{self.what} env {e} t {t}"
                if a.kind != abi.AGENT_NONE:
                    H.assert_close_vec(act[t, e], oa[t], w + " act")
                    assert H.close(rew[t, e], orw[t]) and done[t, e] == od[t], w
                H.assert_close_vec(obs[t, e], oo[t], w + " obs")
                if info is not None and a.kind != abi.AGENT_NONE:          # (no env step, no info row)
                    H.assert_close_vec(info[t, e], oi[t], w + " info")
        self.last_rew, self.last_done = rew, done
        return f"rollout_{how}({T})"

    # ---- checks after every call ---------------------------------------------------------------------------------------------
    def check(self, kind):
        import torch

        from rl4mm_b200 import parallel
        from test_gpu_parity import compare_books

        sim = self.sim
        st = sim.state()
        sd = sim.state_dev()
        assert np.array_equal(sd.cpu().numpy().reshape(-1), st.view(np.uint8)), self.what      # (bytes: NaN prices compare equal)
        assert np.array_equal(sim.errors(), st["err"]), self.what
        if getattr(self, "host_state", None) is not None:
            assert np.array_equal(self.host_state.view(np.uint8), st.view(np.uint8)), self.what
            self.host_state = None
        if getattr(self, "last_rew", None) is not None:
            rew = torch.as_tensor(self.last_rew, device="cuda")
            done = torch.as_tensor(self.last_done, device="cuda")
            a, b = parallel.episode_stats(rew, done, st).cpu().numpy(), parallel.episode_stats_dev(rew, done, sd).cpu().numpy()
            assert np.array_equal(a, b, equal_nan=True), self.what
        for e, o in enumerate(self.oracles):
            w = f"{self.what} env {e}"
            if self.excluded[e]:
                continue
            if H.capacity_excluded(st["err"][e], o, self.cfg, w):
                self.excluded[e] = True
                continue
            os_ = o.state()
            for f in FIELDS:
                assert np.array_equal(st[f][e], os_[f]), (w, f, st[f][e], os_[f])
            assert H.close(st["cash"][e], os_["cash"]) and H.close(st["price"][e], os_["price"]), w
            compare_books(sim, e, o, w)
            if kind == "replay" and self.cfg.fill_log_capacity:
                assert H.canon_fills(sim.fills(e)) == H.canon_fills(o.fills()), w
            if int(os_["err"]) & DEATH_BITS:
                self.excluded[e] = True
            self.checked += 1

    def run(self, n_calls=30):
        self.has_reset = False
        self.what = f"seed {self.seed}: reset"
        self.reset(False, all_envs=True)
        self.check("reset")
        history = []
        for i in range(n_calls):
            r = self.rng.random()
            kind = "other"
            self.what = f"seed {self.seed} after [{', '.join(history[-6:])}] call {i}"
            if r < 0.08:
                name = self.reset(False)
            elif r < 0.16:
                name = self.reset(True)
            elif r < 0.40:
                name, kind = self.replay(str(self.rng.choice(["replay", "replay", "replay_host", "forward_step"])))
            elif r < 0.52:
                name = self.process_orders()
            elif r < 0.60:
                name = self.set_book()
            elif r < 0.72:
                name = self.step(host=bool(self.rng.random() < 0.5))
            else:
                name = self.rollout(str(self.rng.choice(["plain", "info", "agents"])))
            self.what += f" {name}"
            history.append(name)
            self.check(kind)
        self.sim.close()


@pytest.mark.replay_path
@pytest.mark.parametrize("seed", range(SEED0, SEED0 + N_CASES))
def test_random_call_sequence(seed, kernel_family):
    p = Program(seed)
    p.run()
    assert p.checked > 0


def test_replay_host_reads_exactly_its_steps(kernel_family):
    """A stream whose device message array is all zeros, driven only through lobsim_replay_host with the true segment of each call:
    a message read outside the uploaded segment would be a zero record (BAD_VOLUME) or a different book."""
    from oracle.oracle import Oracle
    from test_gpu_parity import compare_books, make_sim

    s = synthetic.generate(synthetic.SynthConfig(seed=31, n_msgs=40_000, duration_s=100, n_levels=10, target_orders=80))
    zero = synthetic.generate(synthetic.SynthConfig(seed=31, n_msgs=40_000, duration_s=100, n_levels=10, target_orders=80))
    zero.msgs[:] = np.zeros(1, abi.MSG_DTYPE)
    kw = dict(n_levels=10, outer_levels=5, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32)
    starts = np.array([10, 20, 50], np.int32)
    sim = make_sim(abi.default_cfg(n_envs=len(starts), **kw), [zero])
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in starts]
    sim.reset_book(0, starts)
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    now = starts.copy()
    for k in (1, 3, 10, 57, 1, 200, 0, 7):
        first, last = int(s.step_off[now.min()]), int(s.step_off[now.max() + k])
        out = np.zeros(len(starts), abi.ENV_STATE_DTYPE)
        sim.replay_host(0, s.msgs[first:last].copy(), first, k, out)
        now += k
        assert np.array_equal(out.view(np.uint8), sim.state().view(np.uint8))
        for e, o in enumerate(oracles):
            o.replay(k)
            os_ = o.state()
            assert out["err"][e] == 0 and os_["err"] == 0, (k, e, out["err"][e])
            for f in FIELDS:
                assert np.array_equal(out[f][e], os_[f]), (k, e, f)
            compare_books(sim, e, o, f"replay_host {k} env {e}")
    sim.close()


def test_step_host_equals_step(kernel_family):
    """Two identical handles, one stepped through lobsim_step and one through lobsim_step_host with the same actions: bit-identical
    outputs and states."""
    import torch

    from test_gpu_parity import make_sim

    rng = np.random.default_rng(5)
    s = _streams(rng, 1)[0]
    kw = _cfg_kw(rng)
    kw["episode_steps"] = 25
    n = 7
    a_sim, b_sim = (make_sim(abi.default_cfg(n_envs=n, **kw), [s]) for _ in range(2))
    starts = np.array([30, 40, 50, 60, 70, 80, 90], np.int32)
    a_sim.reset(0, starts)
    b_sim.reset(0, starts)
    ad, od = abi.action_dim(a_sim.cfg), abi.obs_dim(a_sim.cfg)
    for t in range(40):
        act = rng.uniform(0.2, 6.0, size=(n, ad))
        oa, ra, da = (x.cpu().numpy() for x in a_sim.step(torch.tensor(act, device="cuda")))
        ob, rb, db = np.zeros((n, od)), np.zeros(n), np.zeros(n, np.uint8)
        b_sim.step_host(act, ob, rb, db)
        assert np.array_equal(oa, ob, equal_nan=True) and np.array_equal(ra, rb, equal_nan=True) and np.array_equal(da, db), t
        assert np.array_equal(a_sim.state().view(np.uint8), b_sim.state().view(np.uint8)), t
    a_sim.close()
    b_sim.close()


def test_replay_after_process_orders_tracks_the_agent_orders(kernel_family):
    """After a reset_book of every env no agent order can rest, and replay may take the untracked fast path; agent orders placed by
    lobsim_process_orders must switch it off again, or their fills would leave the agent book stale."""
    from oracle.oracle import Oracle
    from test_gpu_parity import compare_books, make_sim

    s = synthetic.generate(synthetic.SynthConfig(seed=41, n_msgs=40_000, duration_s=100, n_levels=10, target_orders=80, p_sweep=0.02))
    kw = dict(n_levels=10, outer_levels=5, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32)
    starts = np.array([10, 100, 200, 300, 400], np.int32)
    sim = make_sim(abi.default_cfg(n_envs=len(starts), **kw), [s])
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in starts]
    sim.reset_book(0, starts)
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    sim.replay(3)
    st = sim.state()
    orders = []
    for e, o in enumerate(oracles):
        o.replay(3)
        for side in (0, 1):
            for k in range(3):                      # at the touch and one / two ticks behind: filled by the flow of the replay
                px = int(st["best_buy"][e]) - 100 * k if side == 0 else int(st["best_sell"][e]) + 100 * k
                orders.append((e, abi.MSG_LIMIT, side, px, 5 + k, 0, 0, 0))
                o.process_order(abi.MSG_LIMIT, side, px, 5 + k, False, 0)
    sim.process_orders(np.array(orders, abi.ORDER_DTYPE))
    for k in (1, 10, 57):
        sim.replay(k)
        st = sim.state()
        for e, o in enumerate(oracles):
            o.replay(k)
            os_ = o.state()
            for f in FIELDS:
                assert np.array_equal(st[f][e], os_[f]), (k, e, f, st[f][e], os_[f])
            compare_books(sim, e, o, f"replay {k} after process_orders, env {e}")
    assert sum(int(n) for n in np.concatenate(st["n_agent_orders"])) < 6 * len(starts)   # the flow filled some of them
    sim.close()
