"""Randomised differential test: the CUDA path vs the CPU oracle on seeded random streams x random env configurations
(tests/random_cases.py): quote-level ranges, concentration mode, enter_spread, clearing market orders, every feature kind
with random windows and z-score normalisation, every reward kind, resync on/off, thin books that run empty, non-zero
initial inventory, portfolio carry-over across a mid-run reset.  Integer state bit-exact, floats within 1e-6 relative,
error bits identical."""
import numpy as np
import pytest

import parity_helpers as H
import random_cases as R
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu

import os

N_CASES = int(os.environ.get("LOBSIM_RANDOM_CASES", "64"))          # soak runs: LOBSIM_RANDOM_CASES=1000 pytest ...
DEATH_BITS = abi.ERR_EMPTY_BOOK | abi.ERR_NO_SNAPSHOT | abi.ERR_END_OF_STREAM | abi.ERR_BAD_ACTION   # the reference raised: episode over
N_REPLAY_CASES = int(os.environ.get("LOBSIM_RANDOM_REPLAY_CASES", "24"))
SEED0 = int(os.environ.get("LOBSIM_RANDOM_SEED0", "0"))


@pytest.mark.parametrize("seed", range(SEED0, SEED0 + N_CASES))
def test_random_env_case(seed):
    import torch

    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import compare_books, make_sim

    c = R.random_case(seed)
    s = synthetic.generate(c["synth"])
    n, ep = c["n_envs"], c["cfg_kw"]["episode_steps"]
    sim = make_sim(abi.default_cfg(n_envs=n, **c["cfg_kw"]), [s])
    oracles = [Oracle(abi.default_cfg(n_envs=1, **c["cfg_kw"]), s) for _ in range(n)]
    agent, external = c["agent"], c["agent_kind"] == "external"
    # RollingSharpe takes exp(log(aum') - log(aum)) - 1 of AUMs around 1e9..1e12 against returns of 1e-10..1e-12: one ulp of log()
    # moves a return by up to 1e-3 relative.  The device rounds its log / exp correctly (crmath.cuh); the oracle calls glibc's
    # (what numpy does), which is the correctly rounded value except for a few arguments in 1e4 -- so nearly every reward is
    # within 1e-6 (counted below), and the rare others within 1e-3; everything else keeps the 1e-6 tolerance
    sharpe = abi.REWARD_ROLLING_SHARPE in (c["cfg_kw"]["step_reward"].kind, c["cfg_kw"]["terminal_reward"].kind)
    rew_close = (lambda a, b: H.close(a, b, rel=1e-3)) if sharpe else H.close
    n_rew = n_rew_tight = 0
    cfg = abi.default_cfg(n_envs=1, **c["cfg_kw"])
    skipped = set()   # envs whose device book hit a fixed capacity (flagged): with portfolio carry-over they stay different
    for part in range(2):
        starts = (c["starts"] + part * 10).astype(np.int32)
        obs0 = sim.reset(0, starts).cpu().numpy()
        acts = c["actions"][part * ep:(part + 1) * ep]
        # first half of the episode as single steps (lobsim_step), the rest as one fused rollout
        # (a built-in agent: two fused rollouts, its actions are compared as well)
        k = ep // 2
        if external:
            outs = [sim.step(torch.tensor(acts[t], device="cuda")) for t in range(k)]
            obs_a = np.stack([o[0].cpu().numpy() for o in outs]); rew_a = np.stack([o[1].cpu().numpy() for o in outs])
            done_a = np.stack([o[2].cpu().numpy() for o in outs])
            act_a = acts[:k]
        else:
            obs_a, act_a, rew_a, done_a = (x.cpu().numpy() for x in sim.rollout(k, agent))
        obs_b, act_b, rew_b, done_b, info_b = (x.cpu().numpy() for x in sim.rollout(
            ep - k, agent, torch.tensor(acts[k:], device="cuda") if external else None, want_info=True))
        obs, rew, done = np.concatenate([obs_a, obs_b]), np.concatenate([rew_a, rew_b]), np.concatenate([done_a, done_b])
        act = np.concatenate([act_a, act_b])
        st = sim.state()
        for env, o in enumerate(oracles):
            what = f"seed {seed} part {part} env {env}"
            oobs0 = o.reset(int(starts[env]))
            reset_err = int(o.state()["err"])
            oo, oa, orw, od, oi = o.rollout(ep, agent, acts[:, env] if external else None, want_info=True)
            os_ = o.state()
            if H.capacity_excluded(st["err"][env], o, cfg, what):   # fixed capacities are a device-side limit (the oracle is unbounded): flagged, not compared
                skipped.add(env)
            if env in skipped:
                continue
            if not (reset_err & DEATH_BITS):          # (a reset onto an empty book side has no defined observation)
                H.assert_close_vec(obs0[env], oobs0, what + " reset obs")
            assert int(st["err"][env]) == int(os_["err"]), (what, int(st["err"][env]), int(os_["err"]))
            alive = [not (int(oi[t, abi.INFO_FIELDS.index("err")]) & DEATH_BITS) for t in range(ep)]   # outputs after the exception are undefined
            for t in range(ep):
                if t >= k:
                    assert int(info_b[t - k, env, abi.INFO_FIELDS.index("err")]) == int(oi[t, abi.INFO_FIELDS.index("err")]), (what, t)
                if not alive[t]:
                    break
                H.assert_close_vec(act[t, env], oa[t], f"{what} t {t} action")
                H.assert_close_vec(obs[t, env], oo[t], f"{what} t {t} obs")
                assert rew_close(rew[t, env], orw[t]), (what, t, rew[t, env], orw[t])
                n_rew += 1
                n_rew_tight += H.close(rew[t, env], orw[t])
                assert done[t, env] == od[t], (what, t)
                if t >= k:
                    H.assert_close_vec(info_b[t - k, env], oi[t], f"{what} t {t} info")
            compare_books(sim, env, o, what)
            assert st["inventory"][env] == os_["inventory"] and H.close(st["cash"][env], os_["cash"]), what
            assert H.close(st["price"][env], os_["price"]), what
            for f in ("now_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume"):
                assert st[f][env] == os_[f], (what, f, st[f][env], os_[f])
    assert n_rew_tight >= 0.97 * n_rew, (seed, n_rew_tight, n_rew)
    sim.close()


@pytest.mark.fast_only          # the test itself runs both kernel families
@pytest.mark.parametrize("seed", range(SEED0, SEED0 + N_REPLAY_CASES))
def test_random_replay_case(seed, monkeypatch):
    """Pure replay on all four implementations -- the flat order pools (k_replay_flat), the hybrid hot-pool / cold-array book
    (k_replay_hyb, LOBSIM_REPLAY_HYBRID=1 on the layouts that can hold it), the sorted level arrays (k_replay_fast,
    LOBSIM_REPLAY_FLAT=0) and, forced, the general k_advance -- vs the oracle."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import compare_books, make_sim

    c = R.random_replay_case(seed)
    s = synthetic.generate(c["synth"])
    n = c["n_envs"]
    okw = {k: v for k, v in c["cfg_kw"].items() if not k.startswith("max_")}
    cfg = abi.default_cfg(n_envs=n, **c["cfg_kw"])
    for force_general, flat, hyb in (("0", "1", "0"), ("0", "1", "1"), ("0", "0", "0"), ("1", "1", "0")):
        monkeypatch.setenv("LOBSIM_FORCE_GENERAL", force_general)
        monkeypatch.setenv("LOBSIM_REPLAY_HYBRID", hyb)
        monkeypatch.setenv("LOBSIM_REPLAY_FLAT", flat)
        monkeypatch.setenv("LOBSIM_FLAT_BLOBS", flat)
        sim = make_sim(abi.default_cfg(n_envs=n, **c["cfg_kw"]), [s])
        oracles = [Oracle(abi.default_cfg(n_envs=1, **okw), s) for _ in range(n)]
        sim.reset_book(0, c["starts"])
        for o, st in zip(oracles, c["starts"]):
            o.reset_book(int(st))
        for chunk in c["chunks"]:
            sim.replay(chunk)
            st = sim.state()
            for env, o in enumerate(oracles):
                what = f"replay seed {seed} general={force_general} flat={flat} hybrid={hyb} env {env} chunk {chunk}"
                o.replay(chunk)
                os_ = o.state()
                if H.capacity_excluded(st["err"][env], o, cfg, what):   # fixed capacities are a device-side limit: flagged, not compared
                    continue
                assert int(st["err"][env]) == int(os_["err"]), (what, int(st["err"][env]), int(os_["err"]))
                for f in ("now_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume"):
                    assert st[f][env] == os_[f], (what, f, st[f][env], os_[f])
                compare_books(sim, env, o, what)
        sim.close()


def test_per_env_agents_match_oracle_and_sweep_table():
    """lobsim_rollout_agents: one built-in agent per env (parameter sweep) == the oracle run once per (env, agent); then the
    sweep helper of rl4mm_b200/tuning.py on the façade."""
    import ctypes
    from datetime import datetime, timedelta

    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic, tuning
    from rl4mm_b200.agents import FixedActionAgent, Teradactyl
    from rl4mm_b200.features import Inventory, Portfolio, Spread
    from rl4mm_b200.gym import HistoricalOrderbookEnvironment
    from rl4mm_b200.rewards import PnL
    from rl4mm_b200.simulation import DeviceDatabase
    from test_gpu_parity import compare_books, make_sim

    s = synthetic.generate(synthetic.spy_day(seed=21, n_msgs=150_000, duration_s=400))
    feats = [abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000), abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6)]
    kw = dict(n_levels=10, episode_steps=80, warmup_steps=10, features=feats, step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0),
              terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), initial_cash=1e7, max_levels_per_side=64, max_orders_per_side=256)
    rng = np.random.default_rng(3)
    agents = []
    for i in range(11):
        if i % 4 == 3:
            agents.append(abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(*rng.uniform(0.5, 9, 4), 0.0)))
        else:
            agents.append(abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=1, max_inventory=float(rng.choice([100, 1000])),
                                    default_kappa=float(rng.uniform(3, 10)), default_omega=float(rng.uniform(0.2, 0.8)),
                                    max_kappa=float(rng.uniform(10, 14)), exponent=float(rng.choice([1.0, 2.0]))))
    starts = (rng.integers(2, 300, size=len(agents)) * 10).astype(np.int32)
    sim = make_sim(abi.default_cfg(n_envs=len(agents), **kw), [s])
    sim.reset(0, starts)
    obs, act, rew, done, info = (x.cpu().numpy() for x in sim.rollout(80, agents, want_info=True))
    for env, ag in enumerate(agents):
        o = Oracle(abi.default_cfg(n_envs=1, **kw), s)
        o.reset(int(starts[env]))
        oo, oa, orw, od, oi = o.rollout(80, ag, want_info=True)
        for t in range(80):
            H.assert_close_vec(act[t, env], oa[t], f"env {env} t {t} action")
            H.assert_close_vec(obs[t, env], oo[t], f"env {env} t {t} obs")
            H.assert_close_vec(info[t, env], oi[t], f"env {env} t {t} info")
            assert H.close(rew[t, env], orw[t]) and done[t, env] == od[t]
        compare_books(sim, env, o, f"per-env agent {env}")
    sim.close()

    day = datetime(2019, 1, 2)
    db = DeviceDatabase()
    db.add_stream("SPY", day, s)
    grid = tuning.teradactyl_grid(500, [4.0, 8.0], [0.3, 0.5], [12.0], inventory_index=1) + [FixedActionAgent(np.array([1.0, 2.0, 1.0, 2.0]))]
    env = HistoricalOrderbookEnvironment(
        features=[Spread(), Inventory()], ticker="SPY", episode_length=timedelta(seconds=8), min_date=day, max_date=day,
        min_start_timedelta=timedelta(hours=9, minutes=30, seconds=5), max_end_timedelta=timedelta(hours=9, minutes=36),
        initial_portfolio=Portfolio(inventory=0, cash=10**7), per_step_reward_function=PnL(), terminal_reward_function=PnL(),
        n_levels=10, database=db, n_envs=len(grid) * 6, max_levels_per_side=64, max_orders_per_side=256, seed=5)
    table = tuning.sweep_agents(env, grid)
    assert len(table) == len(grid) and all(r["episodes"] == 6 and np.isfinite(r["episode_reward_mean"]) for r in table)
    starts2 = env.episode_start_steps.reshape(len(grid), 6)
    assert (starts2 == starts2[0]).all()                      # every agent saw the same six episodes
    assert len({round(r["episode_reward_mean"], 6) for r in table}) > 1


HYBRID_STRESS = {
    # queues far longer than the 128-order pool at very few prices: the best level cannot become hot (enter fails / bails)
    "long_queues": dict(geom_p=0.6, max_offset_ticks=2, target_orders=700, mean_queue=12, p_sweep=0.01, no=1024),
    # a book around the cold capacity of the 128/512/64 layout (256 cold + 128 hot orders per side): bail on a full cold part
    "cold_full": dict(geom_p=0.1, max_offset_ticks=70, target_orders=760, mean_queue=4, p_sweep=0.0005, no=512),
    # many sweeps through several levels: the pool runs empty inside an execution and is refilled from the cold levels
    "sweeps": dict(geom_p=0.12, max_offset_ticks=70, target_orders=500, mean_queue=1, p_sweep=0.05, no=1024),
    # everything near the touch: the pool fills up and spills its worst level again and again
    "spills": dict(geom_p=0.5, max_offset_ticks=12, target_orders=400, mean_queue=12, p_sweep=0.002, no=1536),
}


@pytest.mark.fast_only
@pytest.mark.parametrize("name", sorted(HYBRID_STRESS))
def test_hybrid_book_stress(name, monkeypatch):
    """k_replay_hyb (book_hybrid.cuh) on streams shaped to hit its conversions: hot <-> cold level moves, pool full, cold part
    full, a best level longer than the pool.  Books, trackers and error flags vs the oracle after every chunk."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic
    from test_gpu_parity import compare_books, make_sim

    k = HYBRID_STRESS[name]
    sc = synthetic.SynthConfig(seed=77, n_msgs=120_000, duration_s=120, n_levels=50, mid0=2_000_000, p_limit=0.40, p_cancel=0.2,
                               p_delete=0.3, p_exec=0.1, geom_p=k["geom_p"], init_levels=55, mean_queue=k["mean_queue"],
                               target_orders=k["target_orders"], max_offset_ticks=k["max_offset_ticks"], p_sweep=k["p_sweep"])
    s = synthetic.generate(sc)
    monkeypatch.setenv("LOBSIM_FORCE_GENERAL", "0")
    monkeypatch.setenv("LOBSIM_REPLAY_FLAT", "1")
    monkeypatch.setenv("LOBSIM_REPLAY_HYBRID", "1")
    n = 4
    kw = dict(n_levels=50, outer_levels=20, resync=1)
    sim = make_sim(abi.default_cfg(n_envs=n, max_levels_per_side=128, max_orders_per_side=k["no"], **kw), [s])
    assert sim.kernel_path == "fast"
    oracles = [Oracle(abi.default_cfg(n_envs=1, **kw), s) for _ in range(n)]
    starts = np.array([0, 100, 300, 500], np.int32)
    sim.reset_book(0, starts)
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    cfg = abi.default_cfg(n_envs=1, max_levels_per_side=128, max_orders_per_side=k["no"], **kw)
    compared = excluded = 0
    for chunk in (1, 9, 90, 250, 250):
        sim.replay(chunk)
        st = sim.state()
        for env, o in enumerate(oracles):
            what = f"hybrid stress {name} env {env} chunk {chunk}"
            o.replay(chunk)
            os_ = o.state()
            if H.capacity_excluded(st["err"][env], o, cfg, what):
                excluded += 1
                continue
            assert int(st["err"][env]) == int(os_["err"]), (what, int(st["err"][env]), int(os_["err"]))
            for f in ("now_step", "min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume"):
                assert st[f][env] == os_[f], (what, f, st[f][env], os_[f])
            compare_books(sim, env, o, what)
            compared += 1
    assert compared >= 8 and compared + excluded == 20, (name, compared, excluded)
    print(f"hybrid stress {name}: {compared} comparisons, {excluded} legitimately excluded (capacity flagged, oracle over capacity)")
    sim.close()
