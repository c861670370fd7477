"""The rolling z-score (Feature.normalise) without a GPU: the oracle against scipy at long windows, the constant-window outcomes
the GPU tests rely on, the exact reference itself, and the depth of the device's pairwise-sum stack at the longest window the
ABI accepts."""
import math
import re
from pathlib import Path

import numpy as np
import pytest

import zscore_reference as Z
from rl4mm_b200 import abi

ROOT = Path(__file__).resolve().parent.parent


def _z_series(raw, maxlen):
    """scipy_z of the reference's history after each update of the clamped values ``raw``."""
    h = np.concatenate([[raw[0] + 1e-06], raw])
    return np.array([Z.scipy_z(h[max(0, u + 2 - maxlen):u + 2]) for u in range(len(raw))])


def test_oracle_matches_scipy_at_long_windows():
    """oracle/lob_oracle.c feature_normalise (an O(n) restatement of scipy) against scipy itself, bit for bit on every update,
    for PRICE and SPREAD histories of 129 to 20 000 entries over 25 000 steps (the long ring is filled and then evicted from),
    and after a reset into a second episode (the history is cleared)."""
    from oracle.oracle import Oracle
    from rl4mm_b200 import synthetic

    s = synthetic.generate(synthetic.SynthConfig(seed=3, n_msgs=3_000_000, duration_s=3000, n_levels=10, mid0=4_000_000))
    lens = (129, 300, 1000, 20_000)
    raw = [abi.feature(abi.FEAT_PRICE, 0, 100_000, 0, 1e8), abi.feature(abi.FEAT_SPREAD, 0, 100_000, 0, 5000)]
    nrm = [abi.feature(f.kind, 0, 100_000, f.min_value, f.max_value, norm_len=L) for L in lens for f in raw]
    steps = (25_000, 1_500)

    def run(feats):
        cfg = abi.default_cfg(n_envs=1, n_levels=10, episode_steps=steps[0], warmup_steps=10, features=feats,
                              step_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0), terminal_reward=abi.Reward(abi.REWARD_PNL, 0, 0.0))
        o = Oracle(cfg, s)
        out = []
        for start, T in zip((200, 26_000), steps):
            obs0 = o.reset(start)
            obs = o.rollout(T, abi.Agent(kind=abi.AGENT_EXTERNAL), np.zeros((T, o.action_dim)))[0]
            out.append(np.concatenate([obs0[None], obs]))
        return out

    raw_eps, z_eps = run(raw), run(nrm)
    n_nan = 0
    for r, z in zip(raw_eps, z_eps):
        for i, L in enumerate(lens):
            for j in range(2):
                want = _z_series(r[:, j], L)
                got = z[:, 2 * i + j]
                bad = [u for u in range(len(want)) if not Z.same_bits(got[u], want[u])]
                assert not bad, (L, j, bad[:5], got[bad[0]], want[bad[0]])
                n_nan += int(np.isnan(want).sum())
    assert n_nan > 0          # the spread sits on one tick for long stretches: constant windows (NaN) are part of the run


# scipy's z of the last entry of a constant window [c] * n: the pairwise mean is off by an ulp or more for some (c, n), which
# turns the NaN of an exactly constant window into -1 or +1 (tests/test_gpu_zscore.py replays these windows on the device)
CONSTANT_WINDOWS = {
    (4e6 + 0.1, 128): -1.0, (4e6 + 0.1, 129): math.nan, (4e6 + 0.1, 136): -1.0, (4e6 + 0.1, 1025): -1.0, (4e6 + 0.1, 20_000): math.nan,
    (0.1, 128): math.nan, (0.1, 129): math.nan, (0.1, 136): 1.0, (0.1, 1025): -1.0, (0.1, 20_000): math.nan,
}


@pytest.mark.parametrize("c,n", sorted(CONSTANT_WINDOWS))
def test_constant_window_outcomes(c, n):
    assert Z.same_bits(Z.scipy_z([c] * n), CONSTANT_WINDOWS[(c, n)])


def test_pairwise_restatement_matches_numpy():
    """The restated split rule (zscore_reference.np_pairwise_sum, the one the stack-depth test below counts) is numpy's: bit for
    bit against np.add.reduce at the leaf and split boundaries, on data whose sum depends on the order."""
    rng = np.random.default_rng(11)
    for n in (1, 2, 7, 8, 9, 15, 16, 17, 127, 128, 129, 135, 136, 137, 255, 256, 257, 1000, 1025, 4097, 20_000):
        a = rng.normal(0, 1, n) * 10.0 ** rng.integers(-8, 9, n)
        assert Z.same_bits(Z.np_pairwise_sum(a), float(np.add.reduce(a))), n
    assert Z.same_bits(Z.np_pairwise_sum(np.array([-0.0] * 5)), -0.0)


def test_exact_z_agrees_with_scipy():
    """exact_z against scipy within 1 eps * kappa on well-conditioned windows (scipy's own error is below that there)."""
    rng = np.random.default_rng(5)
    worst = 0.0
    for n in (2, 3, 8, 100, 129, 1000, 3000):
        for loc, scale in ((0.0, 1.0), (4e6, 1.0), (100.0, 1e-3)):
            w = rng.normal(loc, scale, n)
            z, sd, mean = Z.exact_z(w)
            k = Z.kappa(w[-1], z, sd, mean)
            worst = max(worst, abs(Z.scipy_z(w) - z) / (Z.EPS * k))
    assert worst <= 1.0, worst
    assert math.isnan(Z.exact_z([3.0, 3.0])[0]) and Z.exact_z([1.0, 3.0])[:2] == (1.0, 1.0)


def _define(path: Path, name: str) -> int:
    m = re.search(r"#define\s+" + name + r"\s+(\d+)", path.read_text())
    assert m, f"{name} is not defined in {path.name}"
    return int(m.group(1))


def _max_frames(n_max: int) -> int:
    """Frames the explicit post-order stack of csrc/env.cuh np_pairwise_sum_ring holds at once for some n <= n_max: one per
    level of the split tree, the leaf (n <= 128) included.  Every n, not only n_max: the larger half n - (n/2 - n/2 % 8) is not
    monotonic in n."""
    frames = np.ones(n_max + 1, np.int8)
    lo = 129
    while lo <= n_max:
        hi = min(n_max + 1, 2 * lo - 16)         # both halves of every n < hi are < lo: already known
        n = np.arange(lo, hi)
        n2 = n // 2 - (n // 2) % 8
        frames[lo:hi] = 1 + np.maximum(frames[n2], frames[n - n2])
        lo = hi
    return int(frames.max())


def test_pairwise_stack_fits_the_longest_window():
    """A constant or noise-dominated window is summed in numpy's order through an explicit stack of NP_PAIRWISE_STACK frames;
    validate_cfg accepts histories of up to LOBSIM_MAX_NORM_LEN entries, and the split tree of every such window fits."""
    n_max = _define(ROOT / "include" / "lobsim.h", "LOBSIM_MAX_NORM_LEN")
    env = ROOT / "rl4mm_b200" / "csrc" / "env.cuh"
    stack = _define(env, "NP_PAIRWISE_STACK")
    assert re.search(r"norm_len\s*>\s*LOBSIM_MAX_NORM_LEN", (ROOT / "rl4mm_b200" / "csrc" / "lobsim.cu").read_text())
    body = env.read_text().split("np_pairwise_sum_ring(", 1)[1].split("\n}\n", 1)[0]
    decl = re.search(r"int f_off\[(\w+)\], f_n\[(\w+)\], f_stage\[(\w+)\]; double f_left\[(\w+)\];", body)
    assert decl and set(decl.groups()) == {"NP_PAIRWISE_STACK"}, decl
    assert [_max_frames(n) for n in (128, 129, 2_097_151, 4_194_311)] == [1, 2, 16, 17]
    assert _max_frames(n_max) <= stack, (n_max, _max_frames(n_max), stack)
