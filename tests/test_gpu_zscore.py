"""The rolling z-score of the env kernels (csrc/env.cuh feature_normalise: Feature.normalise, scipy.stats.zscore(history)[-1]
over a deque(maxlen=max_norm_len)) at the window lengths users run -- above the 128-entry leaf of numpy's pairwise sum, where
np_pairwise_sum_ring splits -- against scipy itself (tests/zscore_reference.py), not against the oracle:

* constant and noise-dominated windows, where scipy's answer (NaN or +-1) is its rounding error: bit for bit at every step;
* real feature series on twin runs (normalisation off / on, identical actions): bit for bit in the NaN, constant and noise
  regimes, within NORMAL_C * eps * kappa of the exact z-score and of scipy in the normal regime;
* the features that feed their normalised value back into their own recurrence, against the oracle.

Every episode runs its first half through lobsim_step and the rest through one fused rollout, and a reset clears the histories
before the second episode."""
import functools

import numpy as np
import pytest

import parity_helpers as H
import zscore_reference as Z
from rl4mm_b200 import abi

pytestmark = pytest.mark.gpu

DEVICE = "cuda"
STEP_US = 100_000
CONSTANTS = (0.1, 0.7, 1 / 3, 4e6 + 0.1, 123456.789, 987654.321, 2.2e-9)
LENS = (1, 2, 7, 8, 9, 127, 128, 129, 135, 136, 137, 255, 256, 257, 1000, 1025, 4097)
LONG = 20_000
PNL = abi.Reward(abi.REWARD_PNL, 0, 0.0)


@functools.lru_cache(maxsize=1)
def _stream():
    from rl4mm_b200 import synthetic

    return synthetic.generate(synthetic.SynthConfig(seed=3, n_msgs=2_600_000, duration_s=2600, n_levels=10, mid0=4_000_000))


def _cfg(feats, n_envs, episode_steps, warmup_steps):
    return abi.default_cfg(n_envs=n_envs, n_levels=10, episode_steps=episode_steps, warmup_steps=warmup_steps, features=feats,
                           step_reward=PNL, terminal_reward=PNL, initial_cash=1e9, max_levels_per_side=128,
                           max_orders_per_side=1024)


def _episodes(cfg, starts, steps, actions):
    """Observations [T + 1, n_envs, obs_dim] of each episode (the reset observation first) from the device; each episode
    runs its first half as single steps and the rest as one fused rollout."""
    import torch

    from test_gpu_parity import make_sim

    sim = make_sim(cfg, [_stream()])
    agent = abi.Agent(kind=abi.AGENT_EXTERNAL)
    out = []
    for st, T, acts in zip(starts, steps, actions):
        obs = [sim.reset(0, np.asarray(st, np.int32)).cpu().numpy()[None]]
        k = T // 2
        obs += [sim.step(torch.tensor(acts[t], device=DEVICE))[0].cpu().numpy()[None] for t in range(k)]
        obs.append(sim.rollout(T - k, agent, torch.tensor(acts[k:], device=DEVICE))[0].cpu().numpy())
        out.append(np.concatenate(obs))
    assert not np.any(sim.state()["err"]), sim.state()["err"]
    sim.close()
    return out


# ---- a. constant and noise-dominated windows -------------------------------------------------------------------------
def _constant_window(c, n, offset):
    """[c + 1e-06, c, ..., c] (n entries) when ``offset``, else [c] * n."""
    return ([c + 1e-06] if offset else []) + [c] * (n - offset)


@functools.lru_cache(maxsize=None)
def _constant_want(c, n, offset):
    """scipy's z of the window, its regime, and the normal-regime tolerance."""
    w = _constant_window(c, n, offset)
    zs, reg = Z.scipy_z(w), Z.regime(w)
    if reg != "normal":
        return zs, reg, 0.0
    ze, sd, mean = Z.exact_z_counts([(c + 1e-06, 1), (c, n - 1)] if offset else [(c, n)], c)
    return zs, reg, Z.NORMAL_C * Z.EPS * Z.kappa(c, ze, sd, mean)


def _check_constant(obs, cases, what):
    """obs[u] is the normalised feature after update u (u = 0: the last warm-up step, the reset observation): the history holds
    c + 1e-06 and u + 1 copies of c, the last L of them.  Bit for bit except in the normal regime (a growing window of a small
    c), where the device keeps running sums."""
    for j, (c, L) in enumerate(cases):
        for u in range(obs.shape[0]):
            k = u + 2
            zs, reg, tol = _constant_want(c, min(k, L), k <= L)
            for env in range(obs.shape[1]):
                got = obs[u, env, j]
                assert Z.same_bits(got, zs) if reg != "normal" else abs(got - zs) <= tol, (what, reg, c, L, u, env, got, zs)


def _run_constant(cases, what):
    feats = [abi.feature(abi.FEAT_PRICE, 0, STEP_US, c, c, norm_len=L) for c, L in cases]
    T = max(L for _, L in cases) + 50
    cfg = _cfg(feats, 2, T, 10)
    for obs in _episodes(cfg, ([200, 5000], [1200, 300]), (T, T), [np.zeros((T, 2, 4))] * 2):
        _check_constant(obs, cases, what)


CONSTANT_CASES = [(c, L) for L in LENS for c in CONSTANTS]
CONSTANT_CHUNKS = [CONSTANT_CASES[i:i + abi.MAX_FEATURES] for i in range(0, len(CONSTANT_CASES), abi.MAX_FEATURES)]


@pytest.mark.parametrize("chunk", range(len(CONSTANT_CHUNKS)))
def test_constant_windows(chunk):
    """PRICE clamped to min == max == c: the history grows through [c + 1e-06, c, ...] (the noise regime for large c, the
    normal one for small c) to L entries, then holds [c] * L (the constant regime)."""
    _run_constant(CONSTANT_CHUNKS[chunk], f"constant chunk {chunk}")


@pytest.mark.fast_only
def test_constant_windows_long(monkeypatch):
    """The same at 20 000 entries (a 7-level split tree), on the straight-line kernel and on the general one."""
    cases = [(c, LONG) for c in CONSTANTS]
    _run_constant(cases, "constant long fast")
    monkeypatch.setenv("LOBSIM_FORCE_GENERAL", "1")
    _run_constant(cases, "constant long general")


# ---- b. real feature series, twin runs ---------------------------------------------------------------------------------
CLAMP_WIDTHS = (1e-3, 0.05, 0.2, 2.0)


def _twin_features(c):
    """Features whose normalised value does not feed back (all updated every step); PRICE clamped to [c, c + d] walks its
    windows across the device's 1e-8 switch between the normal and the noise-dominated regime."""
    return [abi.feature(abi.FEAT_SPREAD, 0, STEP_US, 0, 5000), abi.feature(abi.FEAT_PRICE, 0, STEP_US, 0, 1e8),
            abi.feature(abi.FEAT_BOOK_IMBALANCE, 0, STEP_US, -1, 1), abi.feature(abi.FEAT_PRICE_MOVE, 10, STEP_US, -1e4, 1e4),
            abi.feature(abi.FEAT_PRICE_RANGE, 5, STEP_US, 0, 1e4),
            abi.feature(abi.FEAT_TRADE_DIR_IMBALANCE, 20, STEP_US, -1, 1, iparam=0),
            abi.feature(abi.FEAT_TRADE_VOL_IMBALANCE, 20, STEP_US, -1, 1, iparam=1),
            abi.feature(abi.FEAT_TIME_OF_DAY, 0, STEP_US, 0, 21_599, iparam=21_600),
            abi.feature(abi.FEAT_INVENTORY, 0, STEP_US, -1e6, 1e6)] + \
           [abi.feature(abi.FEAT_PRICE, 0, STEP_US, c, c + d) for d in CLAMP_WIDTHS]


def _check_twin(raw, z, L, what, n_exact):
    """raw[u], z[u]: the clamped value and its z-score after update u (u = 0: the first step; warm-up 0).  Returns the counts of
    steps per regime and the worst normal-regime error in eps * kappa."""
    counts = {"nan": 0, "constant": 0, "noise": 0, "normal": 0}
    worst = 0.0
    h = np.concatenate([[raw[0] + 1e-06], raw])
    normal = []
    for u in range(len(raw)):
        w = h[max(0, u + 2 - L):u + 2]
        reg = Z.regime(w)
        counts[reg] += 1
        zs = Z.scipy_z(w)
        if reg != "normal":
            assert Z.same_bits(z[u], zs), (what, reg, u, z[u], zs)
            continue
        mean, sd = Z.numpy_moments(w)
        k = Z.kappa(w[-1], zs, sd, mean)
        assert abs(z[u] - zs) <= Z.NORMAL_C * Z.EPS * k, (what, "vs scipy", u, z[u], zs, abs(z[u] - zs) / (Z.EPS * k))
        normal.append(u)
    for u in normal[::max(1, len(normal) // n_exact)]:
        w = h[max(0, u + 2 - L):u + 2]
        ze, sd, mean = Z.exact_z(w)
        err = abs(z[u] - ze) / (Z.EPS * Z.kappa(w[-1], ze, sd, mean))
        worst = max(worst, err)
        assert err <= Z.NORMAL_C, (what, "vs exact", u, z[u], ze, err)
    return counts, worst


def _run_twin(L, steps, what):
    from oracle.oracle import Oracle

    starts = (15_000 if L < LONG else 200, 10_000)
    o = Oracle(_cfg([abi.feature(abi.FEAT_PRICE, 0, STEP_US, 0, 1e8)], 1, 10, 0), _stream())
    c = float(o.reset(starts[0])[0]) + 0.25                # around the episode's first price
    raw_feats = _twin_features(c)
    z_feats = [abi.feature(f.kind, f.lookback, f.update_us, f.min_value, f.max_value, f.iparam, f.dparam, L) for f in raw_feats]
    rng = np.random.default_rng(L)
    acts = [rng.uniform(0.0, 10.0, size=(T, 1, 4)) for T in steps]      # quotes near the touch: the agent trades
    raws = _episodes(_cfg(raw_feats, 1, max(steps), 0), [[s] for s in starts], steps, acts)
    zs = _episodes(_cfg(z_feats, 1, max(steps), 0), [[s] for s in starts], steps, acts)
    total = {"nan": 0, "constant": 0, "noise": 0, "normal": 0}
    worst = 0.0
    for ep, (r, z) in enumerate(zip(raws, zs)):
        assert np.array_equal(r[0], z[0]), (what, ep)        # warm-up 0: the reset observation is not normalised
        for j in range(len(raw_feats)):
            counts, w = _check_twin(r[1:, 0, j], z[1:, 0, j], L, f"{what} ep {ep} feature {j}", 4 if L == LONG else 20)
            worst = max(worst, w)
            total = {k: total[k] + counts[k] for k in total}
    print(f"{what}: steps per regime {total}, worst normal-regime error {worst:.1f} eps * kappa")
    assert total["noise"] > 0 and total["normal"] > 0, total
    return total


@pytest.mark.parametrize("L", [129, 1000, 4097])
def test_twin_runs(L):
    _run_twin(L, (2 * L + 300, 300), f"twin L={L}")


@pytest.mark.fast_only
def test_twin_runs_long():
    _run_twin(LONG, (LONG + 300, 300), f"twin L={LONG}")


# ---- c. features that normalise their own recurrence -------------------------------------------------------------------
@pytest.mark.parametrize("L", [129, 300, 1000])
def test_stateful_features_vs_oracle(L):
    """VOLATILITY, EPISODE_PROPORTION and AMIHUD_LAMBDA continue their recurrence from the normalised value, so their history
    is only known to an implementation of the whole feature: the device against the oracle (bit for bit against scipy at long
    windows, tests/test_zscore_cpu.py), NaN exactly where the oracle has NaN, the rest within the parity tolerance."""
    from oracle.oracle import Oracle

    feats = [abi.feature(abi.FEAT_VOLATILITY, 20, STEP_US, 0, 1.0, norm_len=L),
             abi.feature(abi.FEAT_EPISODE_PROPORTION, 0, STEP_US, 0, 1, dparam=1.0 / 77, norm_len=L),
             abi.feature(abi.FEAT_AMIHUD_LAMBDA, 12, STEP_US, 0, 1e-3, iparam=3, norm_len=L)]
    steps = (L + 400, 300)
    starts = ([300, 4000, 9000], [12_000, 700, 6000])
    rng = np.random.default_rng(L + 1)
    acts = [rng.uniform(0.0, 10.0, size=(T, 3, 4)) for T in steps]
    cfg = _cfg(feats, 3, max(steps), 30)
    dev = _episodes(cfg, starts, steps, acts)
    oracles = [Oracle(_cfg(feats, 1, max(steps), 30), _stream()) for _ in range(3)]
    n_nan = 0
    for ep, (st, T) in enumerate(zip(starts, steps)):
        for env, o in enumerate(oracles):
            want = np.concatenate([o.reset(st[env])[None], o.rollout(T, abi.Agent(kind=abi.AGENT_EXTERNAL), acts[ep][:, env])[0]])
            for u in range(T + 1):
                H.assert_close_vec(dev[ep][u, env], want[u], f"L={L} ep {ep} env {env} u {u}")
            n_nan += int(np.isnan(want).sum())
    print(f"stateful L={L}: {n_nan} NaN observations")
