"""The capacity error bits against the oracle's high-water marks (oracle.Oracle.peaks).  The device book has fixed capacities,
the oracle's containers are unbounded: a capacity bit must be set exactly when the oracle went over that capacity (no spurious
flag, every set bit justified), in the call in which it first did (the hybrid replay book may instead hold a temporary excess and
end the call equal to the oracle), and until then the device must equal the oracle.  Synthetic streams cross each capacity at
some point of the run; their twins stay under it.  The contract is written next to the error bits in include/lobsim.h."""
import ctypes

import numpy as np
import pytest

import parity_helpers as H
from rl4mm_b200 import abi, synthetic

pytestmark = pytest.mark.gpu

STATE_FIELDS = ("now_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume")


def _synth(seed, n_levels, target_orders, max_offset_ticks, geom_p=0.1, mean_queue=2, p_sweep=0.01, duration_s=140, n_msgs=70_000):
    return synthetic.SynthConfig(seed=seed, n_msgs=n_msgs, duration_s=duration_s, n_levels=n_levels, mid0=2_000_000, p_limit=0.45,
                                 p_cancel=0.15, p_delete=0.3, p_exec=0.1, geom_p=geom_p, init_levels=n_levels + 5, mean_queue=mean_queue,
                                 target_orders=target_orders, max_offset_ticks=max_offset_ticks, p_sweep=p_sweep)


# name: (capacities {levels, orders, agent orders}, stream, does the oracle cross a capacity)
REPLAY_CASES = {
    # the compiled 64/256/32 layout (flat order pools of FLAT_CAP 64 between launches)
    "64_orders": ((64, 256, 32), _synth(1, 10, 300, 30, geom_p=0.2, mean_queue=4), True),
    "64_levels": ((64, 256, 32), _synth(5, 10, 200, 110, geom_p=0.02, mean_queue=1), True),
    "64_under": ((64, 256, 32), _synth(2, 10, 200, 30, geom_p=0.2, mean_queue=4), False),
    # the order capacity crossed while 50-60 levels rest: orders arrive behind the 32 best levels (the rare rest path)
    "64_orders_deep": ((64, 256, 32), _synth(13, 10, 320, 50, geom_p=0.05, mean_queue=3), True),
    # the compiled 128/512/64 layout (the hybrid book's smallest layout)
    "128_orders": ((128, 512, 64), _synth(3, 50, 580, 80, geom_p=0.05), True),
    "128_levels": ((128, 512, 64), _synth(7, 50, 400, 190, geom_p=0.01, mean_queue=1), True),
    "128_under": ((128, 512, 64), _synth(4, 50, 400, 60), False),
    # a triple without a compiled layout: the general runtime-layout kernel in every family
    "96_orders": ((96, 384, 32), _synth(8, 50, 440, 60), True),
    "96_levels": ((96, 384, 32), _synth(9, 50, 300, 150, geom_p=0.02, mean_queue=1), True),
}
STARTS = np.array([0, 150, 300, 450, 600], np.int32)
CALLS = [1] * 40 + [57, 200, 10, 300]      # one grid step per call while the books grow, then long multi-step calls
CASE_CALLS = {"64_orders_deep": [1] * 120 + [200, 300]}


def _cfg(caps, n_levels, **kw):
    nl, no, na = caps
    return abi.default_cfg(n_envs=len(STARTS), n_levels=n_levels, outer_levels=n_levels // 2, resync=1, max_levels_per_side=nl,
                           max_orders_per_side=no, max_agent_orders=na, **kw)


def _replay_and_check(name, family):
    """Replay the case call by call against one oracle per env; returns {env: (index of the first flagged call, its bits)}."""
    from oracle.oracle import Oracle
    from test_gpu_parity import compare_books, make_sim

    caps, sc, _ = REPLAY_CASES[name]
    s = synthetic.generate(sc)
    cfg = _cfg(caps, sc.n_levels)
    sim = make_sim(cfg, [s])
    oracles = [Oracle(_cfg(caps, sc.n_levels), s) for _ in STARTS]
    sim.reset_book(0, STARTS)
    for o, st in zip(oracles, STARTS):
        o.reset_book(int(st))
    first = {}
    for ci, n in enumerate(CASE_CALLS.get(name, CALLS)):
        sim.replay(n)
        st = sim.state()
        for env, o in enumerate(oracles):
            what = f"{name} {family} env {env} call {ci} ({n} steps)"
            o.replay(n)
            ex = H.exceeded_bits(o.peaks(), cfg)
            dev = int(st["err"][env]) & H.CAPACITY_BITS
            assert dev & ~ex == 0, (what, "capacity bits the oracle never earned", dev, ex, o.peaks())
            if env in first:
                assert dev, (what, "capacity bits are sticky")
                continue
            if dev:
                first[env] = (ci, dev)
                continue
            assert not ex or family == "hybrid", (what, "the oracle went over a capacity in this call, the device did not flag", ex, o.peaks())
            assert int(st["err"][env]) == int(o.state()["err"]), what
            os_ = o.state()
            for f in STATE_FIELDS:
                assert st[f][env] == os_[f], (what, f, st[f][env], os_[f])
            compare_books(sim, env, o, what)
    sim.close()
    return first


@pytest.mark.replay_path
@pytest.mark.parametrize("name", sorted(REPLAY_CASES))
def test_replay_capacity_flags_match_oracle_peaks(name, kernel_family):
    first = _replay_and_check(name, kernel_family)
    if REPLAY_CASES[name][2]:
        assert first, (name, "the case is built to cross a capacity")
    else:
        assert not first, (name, first)


@pytest.mark.fast_only
@pytest.mark.parametrize("name", ["64_orders", "64_orders_deep", "64_levels", "128_orders", "128_levels"])
def test_capacity_bits_are_the_same_in_every_family(name, monkeypatch):
    """Per env: the same capacity bits when the device first flags, in every kernel family, and in the same call in the families
    that check at every insertion (the hybrid book flags a level excess when it leaves its form)."""
    got = {}
    for fam, (general, flat, hyb) in {"fast": ("0", "1", "0"), "sorted": ("0", "0", "0"), "general": ("1", "1", "0"),
                                      "hybrid": ("0", "1", "1")}.items():
        monkeypatch.setenv("LOBSIM_FORCE_GENERAL", general)
        monkeypatch.setenv("LOBSIM_REPLAY_FLAT", flat)
        monkeypatch.setenv("LOBSIM_FLAT_BLOBS", flat)
        monkeypatch.setenv("LOBSIM_REPLAY_HYBRID", hyb)
        got[fam] = _replay_and_check(name, fam)
    assert got["fast"], name
    assert got["fast"] == got["sorted"] == got["general"], (name, got)
    for env, (ci, bits) in got["hybrid"].items():
        assert env in got["fast"] and got["fast"][env][1] == bits and ci >= got["fast"][env][0], (name, env, got)


def _fixed(*a):
    return abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(*a, 0.0))


@pytest.mark.parametrize("which", ["over", "under"])
def test_rollout_agent_overflow_flags_match_oracle(which, kernel_family):
    """FixedActionAgent ladders on a deep-queue 50-level book (DESIGN.md section 7, config 5): (1, 2, 1, 2) holds more than 32
    resting agent orders per side after a while, (1, 1, 1, 1) stays under.  One env step per call near the start, then 25."""
    from oracle.oracle import Oracle
    from test_gpu_parity import compare_books, make_sim

    sc = synthetic.heavy_cancel_ticker(seed=3, n_msgs=100_000, duration_s=150)
    sc.target_orders = 180
    s = synthetic.generate(sc)
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(n_levels=50, episode_steps=2000, warmup_steps=0, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e9, max_levels_per_side=64, max_orders_per_side=256,
              max_agent_orders=32)
    starts = np.array([100, 200, 300], np.int32)
    cfg = abi.default_cfg(n_envs=len(starts), **kw)
    sim = make_sim(cfg, [s])
    agent = _fixed(1, 2, 1, 2) if which == "over" else _fixed(1, 1, 1, 1)
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in starts]
    sim.reset(0, starts)
    for o, st in zip(oracles, starts):
        o.reset(int(st))
    flagged = {}
    for ci, T in enumerate([1] * 40 + [25] * 10):
        obs, act, rew, done = (x.cpu().numpy() for x in sim.rollout(T, agent))
        st = sim.state()
        for env, o in enumerate(oracles):
            what = f"{which} {kernel_family} env {env} call {ci}"
            oo, oa, orw, od = o.rollout(T, agent)
            ex = H.exceeded_bits(o.peaks(), cfg)
            dev = int(st["err"][env]) & H.CAPACITY_BITS
            assert dev & ~ex == 0, (what, dev, ex, o.peaks())
            if env in flagged:
                assert dev, what
                continue
            if dev:
                flagged[env] = (ci, dev)
                continue
            assert not ex, (what, "the oracle went over a capacity in this call, the device did not flag", ex, o.peaks())
            for t in range(T):
                H.assert_close_vec(obs[t, env], oo[t], f"{what} t {t} obs")
                assert H.close(rew[t, env], orw[t]), (what, t)
            assert int(st["err"][env]) == int(o.state()["err"]) and st["inventory"][env] == o.state()["inventory"], what
            compare_books(sim, env, o, what)
    if which == "over":
        assert flagged and all(bits == abi.ERR_AGENT_OVERFLOW for _, bits in flagged.values()), flagged
    else:
        assert not flagged, flagged
    sim.close()


def test_fill_log_full_flag_and_truncated_log(kernel_family):
    """A fill log of 8 on a sweep-heavy stream: FILL_LOG_FULL is set exactly when one call recorded more than 8 fills (oracle), the
    log holds the first 8 fills of the call, and the book is unaffected."""
    from oracle.oracle import Oracle
    from test_gpu_parity import compare_books, make_sim

    sc = _synth(11, 10, 120, 20, geom_p=0.3, mean_queue=2, p_sweep=0.05)
    s = synthetic.generate(sc)
    kw = dict(n_levels=10, outer_levels=5, max_levels_per_side=64, max_orders_per_side=256, max_agent_orders=32, fill_log_capacity=8)
    cfg = abi.default_cfg(n_envs=len(STARTS), **kw)
    sim = make_sim(cfg, [s])
    oracles = [Oracle(abi.default_cfg(**kw), s) for _ in STARTS]
    sim.reset_book(0, STARTS)
    for o, st in zip(oracles, STARTS):
        o.reset_book(int(st))
    n_flagged = 0
    for ci, n in enumerate([1] * 30 + [5] * 10 + [40]):
        sim.replay(n)
        st = sim.state()
        for env, o in enumerate(oracles):
            what = f"fill log {kernel_family} env {env} call {ci}"
            o.replay(n)
            want = H.exceeded_bits(o.peaks(), cfg)
            assert want & ~abi.ERR_FILL_LOG_FULL == 0, what
            assert int(st["err"][env]) == int(o.state()["err"]) | want, (what, int(st["err"][env]), want, o.peaks())
            of = o.fills()
            assert H.canon_fills(sim.fills(env)) == H.canon_fills(of[:8]), what
            for f in STATE_FIELDS:
                assert st[f][env] == o.state()[f], (what, f)
            compare_books(sim, env, o, what)
            n_flagged += bool(want)
    assert n_flagged, "the stream is built to overflow the fill log"
    sim.close()
