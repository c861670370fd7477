"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  Everything goes through the C ABI of liblobsim.so.

* against the golden vectors produced by the unmodified reference (tests/golden/),
* against the CPU oracle on seeded synthetic streams (sizes the oracle finishes in seconds),
* size-independent properties at BASELINE.json's full sizes are in tests/test_gpu_fullsize.py.
Integer state (books, fills, inventory) is compared bit-exactly; features / rewards within 1e-6 relative.
"""
import ctypes

import numpy as np
import pytest

import parity_helpers as H
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    return torch


def make_sim(cfg, streams):
    from rl4mm_b200.device import LobSim

    sim = LobSim(cfg, 0)
    for i, s in enumerate(streams):
        sim.load_stream(i, s)
    return sim


class DeviceExchange:
    """Adapter giving one device env the same interface as oracle.Oracle (for the shared fuzz driver)."""

    def __init__(self, cfg, env=0):
        self.cfg, self.env = cfg, env
        self.sim = None
        self._fills = np.zeros(0, abi.FILL_DTYPE)

    def set_stream(self, s):
        self.sim = make_sim(self.cfg, [s])

    def reset_book(self, step):
        self.sim.reset_book(0, step)

    def clear_fills(self):
        self._fills = np.zeros(0, abi.FILL_DTYPE)

    def process_order(self, type, direction, price, volume, is_external, ref):
        o = np.zeros(1, abi.ORDER_DTYPE)
        o[0] = (self.env, type, direction, price, volume, int(is_external), ref & 0xFFFFFFFF, 0)
        fills, refs = self.sim.process_orders(o)
        self._fills = np.concatenate([self._fills, fills])
        return int(refs[0])

    def fills(self):
        return self._fills

    def state(self):
        return self.sim.state(self.env, 1)[0]

    def dump_book(self, side):
        return self.sim.dump_book(self.env, side)

    def dump_agent_orders(self, side):
        return self.sim.dump_agent_orders(self.env, side)


# ---------------------------------------------------------------------------------------------------------------------
#  golden vectors from the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.replay_path
@pytest.mark.parametrize("case_idx", range(4))
def test_fixture_replay_l3_and_fills(case_idx, torch_cuda):
    case = H.load_golden("fixture_replay.json.gz")[case_idx]
    s = H.load_fixture_stream(case["tie_order"])
    n = 6
    sim = make_sim(abi.default_cfg(n_envs=n, outer_levels=case["outer_levels"], fill_log_capacity=512), [s])
    sim.reset_book(0, s.step_of_time(case["start_seconds"]))
    for k, step in enumerate(case["steps"]):
        if k:
            sim.replay(1)
        for env in (0, n - 1):
            for side in (0, 1):
                assert H.canon_book(sim.dump_book(env, side), s.ext_ids) == step["book"][side], (k, env, side)
            if k:
                assert H.canon_fills(sim.fills(env)) == step["fills"], (k, env)
        st = sim.state()
        assert np.all(st["err"] == 0)
        assert np.all(st["min_buy_price"] == step["min_buy"]) and np.all(st["max_sell_price"] == step["max_sell"])


@pytest.mark.replay_path
def test_fixture_replay_in_one_launch(torch_cuda):
    """27 steps fused in one launch == 27 single-step launches (the TMA message pipeline crosses step boundaries)."""
    case = H.load_golden("fixture_replay.json.gz")[0]
    s = H.load_fixture_stream(case["tie_order"])
    sim = make_sim(abi.default_cfg(n_envs=3, outer_levels=case["outer_levels"]), [s])
    sim.reset_book(0, s.step_of_time(case["start_seconds"]))
    sim.replay(27)
    for side in (0, 1):
        assert H.canon_book(sim.dump_book(2, side), s.ext_ids) == case["steps"][27]["book"][side]


@pytest.mark.parametrize("golden,case_idx", H.ENV_GOLDEN_CASES)
def test_env_episodes(golden, case_idx, torch_cuda):
    torch = torch_cuda
    case = H.load_golden(golden)[case_idx]
    s = H.load_fixture_stream("reference")
    n = 3
    sim = make_sim(H.cfg_from_env_case(case, n_envs=n), [s])
    start = s.step_of_time(case["start_seconds"])
    n_rewards = n_tight = 0
    for ep in case["episodes"]:
        obs = sim.reset(0, start).cpu().numpy()
        for env in range(n):
            H.assert_close_vec(obs[env], ep["reset_obs"], "reset obs")
        st = sim.state()
        assert np.all(st["inventory"] == ep["reset_inventory"]) and H.close(st["cash"][0], ep["reset_cash"])
        for side in (0, 1):
            assert H.canon_book(sim.dump_book(n - 1, side), s.ext_ids) == ep["reset_book"][side]
        for k, step in enumerate(ep["steps"]):
            a = torch.tensor([step["action"]] * n, dtype=torch.float64, device="cuda")
            obs, rew, done = (x.cpu().numpy() for x in sim.step(a))
            env = k % n
            for side in (0, 1):
                assert H.canon_book(sim.dump_book(env, side), s.ext_ids) == step["book"][side], (case["name"], k, side)
                got = sorted(map(tuple, H.canon_book(sim.dump_agent_orders(env, side))))
                assert got == sorted(map(tuple, step["agent_book"][side])), (case["name"], k, side)
            assert H.canon_fills(sim.fills(env)) == step["fills"], (case["name"], k)
            st = sim.state()
            assert np.all(st["err"] == 0), st["err"]
            assert np.all(st["inventory"] == step["inventory"]), (case["name"], k)
            assert H.close(st["cash"][env], step["cash"]) and H.close(st["price"][env], step["price"])
            H.assert_close_vec(obs[env], step["obs"], f"{case['name']} step {k} obs")
            assert H.reward_close(rew[env], step), (case["name"], k, rew[env], step["reward"], step.get("bound"))
            n_rewards += 1
            n_tight += H.close(rew[env], step["reward"])
            assert bool(done[env]) == step["done"]
            # identical replicas stay identical (RollingSharpe over a single return is NaN in the reference too)
            assert np.array_equal(obs, np.broadcast_to(obs[0], obs.shape), equal_nan=True)
            assert np.array_equal(rew, np.full_like(rew, rew[0]), equal_nan=True)
    # the correctly rounded log / exp of the device (crmath.cuh) keep nearly every RollingSharpe reward at 1e12 cash within 1e-6
    # of the reference; the analytic bound is needed only where glibc's log is not the correctly rounded value
    assert n_tight >= 0.9 * n_rewards, (case["name"], n_tight, n_rewards)


@pytest.mark.parametrize("case_idx", range(120))
def test_exchange_fuzz(case_idx, torch_cuda):
    from test_oracle_golden import replay_exchange_case

    case = H.load_golden("exchange_fuzz.json.gz")[case_idx]
    replay_exchange_case(DeviceExchange(abi.default_cfg(n_envs=2), env=1), case)


def test_beta_ladders_exact(torch_cuda):
    """Lot sizes of every golden action (scipy.stats.beta.pdf + np.round) on a step with no fills."""
    torch = torch_cuda
    s = H.load_fixture_stream("reference")
    start = s.step_of_time(36000.0)
    checked = 0
    for grp in H.load_golden("beta_ladders.json.gz"):
        cases = grp["cases"]
        n = len(cases)
        cfg = abi.default_cfg(n_envs=n, min_quote_level=0, max_quote_level=grp["quote_levels"],
                              active_volume=grp["active_volume"],
                              concentration=-1.0 if grp["concentration"] is None else grp["concentration"],
                              features=[abi.feature(abi.FEAT_INVENTORY, 0, 100000, -1e6, 1e6)], outer_levels=48,
                              portfolio_carryover=0, fill_log_capacity=64)
        sim = make_sim(cfg, [s])
        sim.reset(0, start)
        st0 = sim.state()
        acts = torch.tensor([c["action"] for c in cases], dtype=torch.float64, device="cuda")
        sim.step(acts)
        for env, c in enumerate(cases):
            if len(sim.fills(env)):
                continue
            bb, bs = int(st0["best_buy"][env]), int(st0["best_sell"][env])
            for side, exp, base, sgn in ((0, c["buy"], bb, -1), (1, c["sell"], bs, +1)):
                got = {int(e["price"]): int(e["volume"]) for e in sim.dump_agent_orders(env, side)}
                want = {base + sgn * 100 * k: v for k, v in enumerate(exp) if v > 0}
                assert got == want, (grp["quote_levels"], c["action"])
            checked += 1
        sim.close()
    assert checked > 500


# ---------------------------------------------------------------------------------------------------------------------
#  CUDA vs CPU oracle on synthetic streams
# ---------------------------------------------------------------------------------------------------------------------
def compare_books(sim, env, oracle, what):
    for side in (0, 1):
        d, o = sim.dump_book(env, side), oracle.dump_book(side)
        assert len(d) == len(o), (what, side, len(d), len(o))
        # agent ids are implementation-defined: compare (price, volume) and the ref of non-agent orders
        assert np.array_equal(d["price"], o["price"]) and np.array_equal(d["volume"], o["volume"]), (what, side)
        da, oa = (d["ref"] & abi.REF_AGENT) != 0, (o["ref"] & abi.REF_AGENT) != 0
        assert np.array_equal(da, oa) and np.array_equal(d["ref"][~da], o["ref"][~oa]), (what, side)
        ad, ao = sim.dump_agent_orders(env, side), oracle.dump_agent_orders(side)
        assert np.array_equal(ad["price"], ao["price"]) and np.array_equal(ad["volume"], ao["volume"]), (what, side)


@pytest.mark.replay_path
@pytest.mark.parametrize("which", ["spy", "heavy"])
def test_synthetic_replay_vs_oracle(which, torch_cuda):
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic

    if which == "spy":
        sc = synthetic.spy_day(seed=11, n_msgs=300_000, duration_s=700)
        cap = dict(max_levels_per_side=64, max_orders_per_side=256)
    else:
        sc = synthetic.heavy_cancel_ticker(seed=5, n_msgs=200_000, duration_s=400)
        cap = dict(max_levels_per_side=128, max_orders_per_side=1536)
    s = synthetic.generate(sc)
    starts = [0, 10, 50, 1000, 2500]  # grid steps on whole seconds
    cfg = abi.default_cfg(n_envs=len(starts), n_levels=sc.n_levels, outer_levels=20, **cap)
    sim = make_sim(cfg, [s])
    sim.reset_book(0, np.array(starts, np.int32))
    oracles = [Oracle(abi.default_cfg(n_levels=sc.n_levels, outer_levels=20), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(st)
    for chunk in (1, 9, 490, 1000):
        sim.replay(chunk)
        st = sim.state()
        for env, o in enumerate(oracles):
            o.replay(chunk)
            os_ = o.state()
            assert st["err"][env] == os_["err"] == 0, (which, env, st["err"][env], os_["err"])
            assert st["now_step"][env] == os_["now_step"]
            for f in ("min_buy_price", "max_sell_price", "best_buy", "best_sell", "best_buy_volume", "best_sell_volume"):
                assert st[f][env] == os_[f], (which, env, chunk, f, st[f][env], os_[f])
            compare_books(sim, env, o, (which, env, chunk))


def rollout_features():
    return [
        abi.feature(abi.FEAT_SPREAD, 0, 100000, 0, 5000),
        abi.feature(abi.FEAT_PRICE_MOVE, 1, 100000, -10000, 10000),
        abi.feature(abi.FEAT_PRICE_MOVE, 10, 1000000, -10000, 10000),
        abi.feature(abi.FEAT_VOLATILITY, 50, 100000, 0, 1.0),
        abi.feature(abi.FEAT_VOLATILITY, 10, 1000000, 0, 1.0),
        abi.feature(abi.FEAT_INVENTORY, 0, 100000, -1e6, 1e6),
        abi.feature(abi.FEAT_EPISODE_PROPORTION, 0, 100000, 0, 1, dparam=100000 / (60 * 1e6)),
        abi.feature(abi.FEAT_TIME_OF_DAY, 0, 60000000, 0, 9, iparam=10),
        abi.feature(abi.FEAT_TRADE_DIR_IMBALANCE, 50, 100000, -1, 1),
        abi.feature(abi.FEAT_TRADE_VOL_IMBALANCE, 50, 100000, -1, 1, iparam=1),
        abi.feature(abi.FEAT_BOOK_IMBALANCE, 0, 100000, -1, 1),
        abi.feature(abi.FEAT_PRICE_RANGE, 5, 500000, 0, 10000),
        abi.feature(abi.FEAT_PRICE, 0, 1000000, 0, 1e8),
    ]


@pytest.mark.parametrize("levels_cap", [64, 128])
@pytest.mark.parametrize("agent_kind", ["fixed", "teradactyl", "external", "random"])
def test_synthetic_rollout_vs_oracle(agent_kind, levels_cap, torch_cuda):
    """Full env path (agent orders, fills, portfolio, features, rewards, resync) on a synthetic SPY-shaped stream.  levels_cap 128
    = the 128/256/64 layout, which the flat form may fill with 128 orders per side (book_flat.cuh); its step / rollout launches run
    on the env kernel k_env_fast, which works on the sorted form only and converts a flat blob on load."""
    torch = torch_cuda
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic

    sc = synthetic.spy_day(seed=3, n_msgs=400_000, duration_s=900)
    s = synthetic.generate(sc)
    warm = 100  # max window: 10 x 1 s = 10 s => 100 steps
    starts = [200, 1000, 3000, 3010]
    kw = dict(n_levels=10, episode_steps=200, warmup_steps=warm, outer_levels=20, features=rollout_features(),
              step_reward=abi.Reward(abi.REWARD_INV_ADJ_PNL, 0, 1e-4), terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0),
              max_levels_per_side=levels_cap, max_orders_per_side=256, max_agent_orders=64,
              market_order_clearing=1 if agent_kind == "teradactyl" else 0,
              market_order_fraction_of_inventory=0.25 if agent_kind == "teradactyl" else 0.0)
    sim = make_sim(abi.default_cfg(n_envs=len(starts), **kw), [s])
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(len(starts))]
    obs_d = sim.reset(0, np.array(starts, np.int32)).cpu().numpy()
    for env, (o, st) in enumerate(zip(oracles, starts)):
        H.assert_close_vec(obs_d[env], o.reset(st), f"reset obs env {env}")
    T = 300
    ad = abi.action_dim(sim.cfg)
    acts = None
    if agent_kind == "fixed":
        agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 2, 1, 2, 0))
    elif agent_kind == "teradactyl":
        agent = abi.Agent(kind=abi.AGENT_TERADACTYL, inventory_index=5, max_inventory=300.0, default_kappa=7.0,
                          default_omega=0.4, max_kappa=12.0, exponent=1.5, market_clearing=1)
    elif agent_kind == "random":   # device RandomAgent (Philox keyed by seed, env, grid step) == its oracle twin, bit for bit
        agent = abi.Agent(kind=abi.AGENT_RANDOM, fixed_action=(ctypes.c_double * 5)(10, 10, 10, 10, 0), reserved=1234)
    else:
        agent = abi.Agent(kind=abi.AGENT_EXTERNAL)
        acts = np.random.default_rng(0).uniform(0, 10, size=(T, len(starts), ad))
    half = T // 2
    for part in range(2):  # two launches: books and feature windows must survive the HBM round trip
        sl = slice(part * half, (part + 1) * half)
        a_in = None if acts is None else torch.tensor(acts[sl], device="cuda")
        obs, act, rew, done = (x.cpu().numpy() for x in sim.rollout(half, agent, a_in))
        for env, o in enumerate(oracles):
            oo, oa, orw, od = o.rollout(half, agent, None if acts is None else acts[sl, env])
            for t in range(half):
                H.assert_close_vec(act[t, env], oa[t], f"{agent_kind} env {env} t {t} action")
                if agent_kind == "random":
                    assert np.array_equal(act[t, env], oa[t]) and np.all(act[t, env] >= 0) and np.all(act[t, env] < 10)
                H.assert_close_vec(obs[t, env], oo[t], f"{agent_kind} env {env} t {part * half + t} obs")
                assert H.close(rew[t, env], orw[t]), (agent_kind, env, t, rew[t, env], orw[t])
                assert done[t, env] == od[t]
            compare_books(sim, env, o, (agent_kind, env, part))
            st, os_ = sim.state(env, 1)[0], o.state()
            assert st["err"] == os_["err"] == 0
            assert st["inventory"] == os_["inventory"] and H.close(st["cash"], os_["cash"])
        if agent_kind == "random":    # envs 2 and 3 start 10 steps apart: different env index => different action streams
            assert not np.array_equal(act[:, 2], act[:, 3]) and not np.array_equal(act[10:, 2], act[:-10, 3])
