"""The replay kernels (k_replay_flat, k_replay_hyb, k_replay_fast, k_advance) and the env kernels on the adversarial streams of
tests/adversarial_streams.py: crossing limits, multi-order and multi-level executions, exact and over-size removals, unknown
and reused refs, churned queues, full flat pools, hybrid hot pools that run empty inside one message, a best level longer than
the hybrid pool, extreme prices and volumes, and EmptyOrderbookError in the middle of a second.  Everything is compared with
the oracle: error bits and now_step exactly, state fields and L3 books exactly, fills field by field."""
import ctypes

import numpy as np
import pytest

import adversarial_streams as A
import parity_helpers as H
from rl4mm_b200 import abi

pytestmark = [pytest.mark.gpu, pytest.mark.replay_path]

STREAMS = [(shape, seed) for shape, sh in A.SHAPES.items() for seed in sh["seeds"]]
CHUNKS = (1, 3, 7, 10, 23, 57)          # ragged: launches start and end part-way through seconds
COMPILED = {(64, 256), (128, 512), (128, 1024)}        # (levels, orders) pairs of the stream shapes with a compiled layout


def _caps(shape, kernel_family):
    """Capacity pairs to run a shape at: deep books also at 128/512, which takes the hybrid book only under LOBSIM_REPLAY_HYBRID."""
    nl, no, _ = A.SHAPES[shape]["caps"]
    return [(nl, no), (128, 512)] if shape == "deep" and kernel_family == "hybrid" else [(nl, no)]


def _sim_and_oracles(s, shape, starts, caps, **kw):
    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim

    nl, no = caps
    kw = dict(kw, max_levels_per_side=nl, max_orders_per_side=no)
    sim = LobSim(A.cfg_for(shape, n_envs=len(starts), **kw), 0)
    sim.load_stream(0, s)
    sim.reset_book(0, np.array(starts, np.int32))
    oracles = [Oracle(A.cfg_for(shape, **kw), s) for _ in starts]
    for o, st in zip(oracles, starts):
        o.reset_book(int(st))
    return sim, oracles


def _assert_fills_equal(d, f, what):
    """Fill records field by field in emission order; of the ref, only whether it names an agent order (agent ids are
    implementation-defined) and the ref of every other order."""
    assert len(d) == len(f), (what, len(d), len(f))
    for name in abi.FILL_DTYPE.names:
        if name != "ref":
            assert np.array_equal(d[name], f[name]), (what, name)
    da, fa = (d["ref"] & abi.REF_AGENT) != 0, (f["ref"] & abi.REF_AGENT) != 0
    assert np.array_equal(da, fa) and np.array_equal(d["ref"][~da], f["ref"][~fa]), (what, "ref")


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
    return st


@pytest.mark.parametrize("shape,seed", STREAMS)
def test_adversarial_replay_matches_oracle(shape, seed, kernel_family):
    """Six books per stream, started on different seconds, replayed to the end of the stream in ragged launches; after every
    launch error bits, now_step (the death step included), trackers, best prices and volumes and L3 books are the oracle's."""
    import torch

    assert torch.cuda.is_available()
    s = A.build(shape, seed)
    starts = [10 * t for t in A.STARTS]
    for caps in _caps(shape, kernel_family):
        sim, oracles = _sim_and_oracles(s, shape, starts, caps, resync=0, outer_levels=2)
        if kernel_family != "general" and caps in COMPILED:
            assert sim.kernel_path == "fast", (caps, sim.kernel_path)
        else:
            assert sim.kernel_path != "fast", (caps, sim.kernel_path)
        _check(sim, oracles, ("reset", caps))
        done, k, flat_seen = 0, 0, False
        while done < s.n_grid_steps:
            chunk = CHUNKS[k % len(CHUNKS)]
            k += 1
            sim.replay(chunk)
            for o in oracles:
                o.replay(chunk)
            done += chunk
            st = _check(sim, oracles, (caps, done, chunk))
            flat_seen |= bool(np.any(st["reserved"][: len(starts)] & 1))
        deaths = int(np.sum((st["err"][: len(starts)] & abi.ERR_EMPTY_BOOK) != 0))
        assert 0 < deaths, "the stream kills at least one of its books (EmptyOrderbookError)"
        assert np.all(st["err"][: len(starts)] & (abi.ERR_EMPTY_BOOK | abi.ERR_END_OF_STREAM))
        if shape == "thin" and kernel_family in ("fast", "hybrid"):
            assert flat_seen, "the thin books ran in the flat form"
        sim.close()


@pytest.mark.parametrize("shape,seed", STREAMS)
def test_adversarial_fill_logged_replay_matches_oracle(shape, seed, kernel_family):
    """A fill log routes the replay to the general k_advance: one step per launch over the seconds of the side sweeps, the hot-pool
    sweeps and the death; the fills of every step are the oracle's, field by field, in emission order."""
    s = A.build(shape, seed)
    starts = [100, 120, 520, 550]
    for caps in _caps(shape, kernel_family):
        sim, oracles = _sim_and_oracles(s, shape, starts, caps, resync=0, outer_levels=2, fill_log_capacity=8192)
        n_fills = 0
        for step in range(60):
            sim.replay(1)
            for o in oracles:
                o.replay(1)
            _check(sim, oracles, (caps, "fill log", step))
            for env, o in enumerate(oracles):
                f = o.fills()
                _assert_fills_equal(sim.fills(env), f, (caps, step, env))
                n_fills += len(f)
        assert n_fills > 1000
        sim.close()


@pytest.mark.parametrize("shape,seed", STREAMS)
def test_adversarial_forward_step_with_resync_matches_oracle(shape, seed, kernel_family):
    """Replay and forward_step interleaved, resync on: the side sweeps leave books thin, so update_outer_levels rewrites them."""
    s = A.build(shape, seed)
    starts = [0, 70, 160, 270]
    for caps in _caps(shape, kernel_family):
        sim, oracles = _sim_and_oracles(s, shape, starts, caps, resync=1, outer_levels=max(1, A.SHAPES[shape]["n_levels"] // 5))
        done, k = 0, 0
        while done < 400:
            kind = "forward" if k % 2 else "replay"
            chunk = (13, 30, 4, 41, 10, 27)[k % 6]
            k += 1
            sim.replay(chunk) if kind == "replay" else sim.forward_step(chunk)
            for o in oracles:
                o.replay(chunk) if kind == "replay" else o.forward_step(chunk)
            done += chunk
            _check(sim, oracles, (caps, kind, done))
        sim.close()


def _rollout_features():
    return [
        abi.feature(abi.FEAT_TRADE_DIR_IMBALANCE, 20, 100_000, -1, 1, iparam=1),
        abi.feature(abi.FEAT_TRADE_VOL_IMBALANCE, 20, 100_000, -1, 1, iparam=1),
        abi.amihud(4, 2, 100_000, 0, 1e-3),
        abi.feature(abi.FEAT_BOOK_IMBALANCE, 0, 100_000, -1, 1),
        abi.feature(abi.FEAT_INVENTORY, 0, 100_000, -1e6, 1e6),
    ]


@pytest.mark.parametrize("agent_kind", ["fixed", "external"])
@pytest.mark.parametrize("shape", ["thin", "deep"])
def test_adversarial_env_rollout_matches_oracle(shape, agent_kind, kernel_family):
    """Env rollouts over the adversarial streams: historical crossing limits and sweeps fill the agent's resting orders.  Two
    episodes per env; obs and rewards within the parity tolerances, inventory, cash, books, agent books and fills exactly."""
    import torch

    from oracle.oracle import Oracle
    from rl4mm_b200.device import LobSim
    from test_gpu_parity import compare_books

    s = A.build(shape, 0)
    nl = {"thin": 64, "deep": 128}[shape]
    no = {"thin": 256, "deep": 1024}[shape]
    kw = dict(n_levels=s.n_levels, episode_steps=60, warmup_steps=30, outer_levels=2, features=_rollout_features(),
              step_reward=abi.Reward(abi.REWARD_INV_ADJ_PNL, 0, 1e-4), terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0),
              max_levels_per_side=nl, max_orders_per_side=no, max_agent_orders=64, enter_spread=1,
              market_order_clearing=1, market_order_fraction_of_inventory=0.5, fill_log_capacity=4096)
    starts = [100, 230, 480, 540]
    sim = LobSim(abi.default_cfg(n_envs=len(starts), **kw), 0)
    sim.load_stream(0, s)
    oracles = [Oracle(abi.default_cfg(**kw), s, env_index=i) for i in range(len(starts))]
    obs_d = sim.reset(0, np.array(starts, np.int32)).cpu().numpy()
    for env, (o, st) in enumerate(zip(oracles, starts)):
        H.assert_close_vec(obs_d[env], o.reset(st), f"reset obs env {env}")
    ad = abi.action_dim(sim.cfg)
    T = 2 * kw["episode_steps"]
    acts = None
    if agent_kind == "fixed":
        agent = abi.Agent(kind=abi.AGENT_FIXED, fixed_action=(ctypes.c_double * 5)(1, 3, 2, 1, 100))
    else:
        agent = abi.Agent(kind=abi.AGENT_EXTERNAL)
        acts = np.random.default_rng(3).uniform(0, 1, size=(T, len(starts), ad)) * np.array([10, 10, 10, 10, 200])[:ad]
    t, n_fills = 0, 0
    for chunk in [1, 9] * (T // 10):
        sl = slice(t, t + chunk)
        a_in = None if acts is None else torch.tensor(acts[sl], device="cuda")
        obs, act, rew, done = (x.cpu().numpy() for x in sim.rollout(chunk, agent, a_in))
        st = sim.state()
        for env, o in enumerate(oracles):
            oo, oa, orw, od = o.rollout(chunk, agent, None if acts is None else acts[sl, env])
            for j in range(chunk):
                H.assert_close_vec(act[j, env], oa[j], f"{shape} {agent_kind} env {env} t {t + j} action")
                H.assert_close_vec(obs[j, env], oo[j], f"{shape} {agent_kind} env {env} t {t + j} obs")
                assert H.close(rew[j, env], orw[j]), (shape, agent_kind, env, t + j, rew[j, env], orw[j])
                assert done[j, env] == od[j], (env, t + j)
            os_ = o.state()
            assert int(st["err"][env]) == int(os_["err"]), (env, t, int(st["err"][env]), int(os_["err"]))
            assert st["inventory"][env] == os_["inventory"] and st["cash"][env] == os_["cash"], (env, t)
            compare_books(sim, env, o, (shape, agent_kind, env, t))
            if chunk == 1:                                   # the fill log holds the fills of the call's last step
                f = o.fills()
                _assert_fills_equal(sim.fills(env), f, (shape, agent_kind, env, t))
                n_fills += len(f)
        t += chunk
    assert n_fills > 0
    sim.close()
