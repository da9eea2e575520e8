"""Reward normalisation of Algo_PPO(normalize_reward=True) (DESIGN.md §4 "Reward normalisation"), no GPU: the option checks of the
constructor (which run before the env is touched) and a float64 restatement of the rule -- the forward running return, the batch
moments of both streams, SB3's RunningMeanStd.update_from_moments and the scale / clip -- checked against SB3's RunningMeanStd and
VecNormalize reward path as written there (SB3 is not a dependency, so its formulas are restated below).
tests/test_reward_norm_gpu.py holds mhppo_reward_moments, mhppo_reward_normalize and the update to this restatement."""
import math
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_grad_clip import _Untouchable  # noqa: E402

RMS0 = np.array([[1e-4, 0.0, 1.0], [1e-4, 0.0, 1.0]])      # (count, mean, var) of each stream at the start
EPS = 1e-8


# ---------------------------------------------------------------------------------------------------------------------
# the restatement

def running_returns(rew, gamma):
    """g_t = gamma * g_{t-1} + r_t over t = 0 .. T-1 of rew [T][CN] (g_{-1} = 0), float64: [T][CN]."""
    rew = np.asarray(rew, dtype=np.float64)
    g, out = np.zeros(rew.shape[1]), np.empty_like(rew)
    for t in range(rew.shape[0]):
        g = gamma * g + rew[t]
        out[t] = g
    return out


def batch_moments(rew, rew_d, route, gamma):
    """(n, sum g, sum g^2) of the continuous stream, then (n, sum x, sum x^2) of the choice stream, over the columns with
    route >= 0: what mhppo_reward_moments writes."""
    on = np.asarray(route) >= 0
    g = running_returns(rew, gamma)[:, on]
    x = np.asarray(rew_d, dtype=np.float64)[on]
    return np.array([g.size, g.sum(), (g * g).sum(), x.size, x.sum(), (x * x).sum()])


def merge(rms, moments):
    """The running state [2][3] after merging the batch moments (SB3's update_from_moments; an empty stream keeps its state)."""
    out = np.array(rms, dtype=np.float64)
    for s in range(2):
        n, s1, s2 = moments[3 * s: 3 * s + 3]
        if not n > 0:
            continue
        mb = s1 / n
        vb = max(s2 / n - mb * mb, 0.0)
        count, mean, var = out[s]
        delta, tot = mb - mean, count + n
        out[s] = (tot, mean + delta * n / tot, (var * count + vb * n + delta * delta * count * n / tot) / tot)
    return out


def scale(r, var, clip):
    """clip(r / sqrt(var + 1e-8), -clip, clip) in float64, rounded to float32 once."""
    x = np.asarray(r, dtype=np.float64) / np.sqrt(var + EPS)
    return np.clip(x, -clip, clip).astype(np.float32)


# SB3 (stable_baselines3/common/running_mean_std.py, vec_env/vec_normalize.py), restated
class RunningMeanStd:
    def __init__(self, epsilon=1e-4):
        self.mean, self.var, self.count = 0.0, 1.0, epsilon

    def update(self, arr):
        self.update_from_moments(np.mean(arr, axis=0), np.var(arr, axis=0), arr.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / tot_count
        self.mean, self.var, self.count = new_mean, m_2 / tot_count, tot_count


class VecNormalizeReward:
    """VecNormalize(norm_obs=False, norm_reward=True): step_wait's reward path."""
    def __init__(self, num_envs, gamma, clip_reward=10.0, epsilon=1e-8):
        self.ret_rms, self.returns = RunningMeanStd(), np.zeros(num_envs)
        self.gamma, self.clip_reward, self.epsilon = gamma, clip_reward, epsilon

    def step(self, rewards, dones):
        self.returns = self.returns * self.gamma + rewards
        self.ret_rms.update(self.returns)
        out = np.clip(rewards / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)
        self.returns[dones] = 0
        return out


def _rollout(T, CN, seed, absent=0.3):
    rng = np.random.default_rng(seed)
    rew = (rng.standard_normal((T, CN)) * 3.0 - 1.0).astype(np.float32)
    rew_d = np.minimum(rng.standard_normal(CN) * 4.0, 0.0).astype(np.float32)
    route = rng.choice(np.array([-1, 0, 1], dtype=np.int8), CN, p=[absent, (1 - absent) / 2, (1 - absent) / 2])
    return rew, rew_d, route


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(np.abs(np.asarray(b)), 1e-300)


# ---------------------------------------------------------------------------------------------------------------------
# 1. option checks

_BASE = dict(num_states_c=13, num_states_d=18)


@pytest.mark.parametrize("opts", [dict(normalize_reward=1), dict(normalize_reward="yes"), dict(normalize_reward=np.bool_(True)),
                                  dict(normalize_reward=None),
                                  dict(normalize_reward=True, clip_reward=True), dict(normalize_reward=True, clip_reward=math.nan),
                                  dict(normalize_reward=True, clip_reward=0), dict(normalize_reward=True, clip_reward=0.0),
                                  dict(normalize_reward=True, clip_reward=-5.0), dict(normalize_reward=True, clip_reward=-math.inf),
                                  dict(normalize_reward=True, clip_reward="10"), dict(normalize_reward=True, clip_reward=[10.0]),
                                  dict(clip_reward=10.0), dict(normalize_reward=False, clip_reward=math.inf)])
def test_options_rejected_before_the_env_is_touched(opts):
    import mhppo_b200 as mh
    with pytest.raises(ValueError):
        mh.Algo_PPO(mh.Model_PPO, _Untouchable(), **_BASE, **opts)


@pytest.mark.parametrize("opts", [{}, dict(normalize_reward=False), dict(normalize_reward=True),
                                  dict(normalize_reward=True, clip_reward=None), dict(normalize_reward=True, clip_reward=5),
                                  dict(normalize_reward=True, clip_reward=0.5), dict(normalize_reward=True, clip_reward=math.inf),
                                  dict(normalize_reward=True, clip_reward=np.float32(10.0))])
def test_options_accepted(opts):
    """An accepted value passes the option checks: the constructor goes on to read the env."""
    import mhppo_b200 as mh
    with pytest.raises(AssertionError, match="touched the env"):
        mh.Algo_PPO(mh.Model_PPO, _Untouchable(), **_BASE, **opts)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the restatement against SB3's

@pytest.mark.parametrize("T,CN", [(1, 8), (7, 33), (80, 1000)])
def test_merge_equals_running_mean_std_on_the_returns(T, CN):
    """Merging a rollout's batch moments equals RunningMeanStd.update on the concatenated returns of the present columns (and on
    the present choice rewards), for two rollouts in a row."""
    gamma = 0.99
    rms = RMS0.copy()
    ref = [RunningMeanStd(), RunningMeanStd()]
    for seed in (1, 2):
        rew, rew_d, route = _rollout(T, CN, seed)
        on = route >= 0
        mom = batch_moments(rew, rew_d, route, gamma)
        assert mom[0] == T * on.sum() and mom[3] == on.sum()
        rms = merge(rms, mom)
        ref[0].update(running_returns(rew, gamma)[:, on].reshape(-1))
        ref[1].update(rew_d[on].astype(np.float64))
        for s in range(2):
            want = np.array([ref[s].count, ref[s].mean, ref[s].var])
            assert rms[s][0] == want[0]
            assert (_rel(rms[s][1:], want[1:]) <= 1e-12).all(), (rms[s], want)


@pytest.mark.parametrize("clip", [10.0, 0.5, math.inf])
def test_one_step_rollouts_equal_vec_normalize(clip):
    """At T = 1 the whole-rollout rule equals SB3's per-step VecNormalize reward path (every rollout is one step and one episode,
    so SB3 resets its returns after each), clip included; present columns are SB3's envs, for both streams."""
    gamma, CN = 0.99, 300
    rms = RMS0.copy()
    rng = np.random.default_rng(5)
    route = rng.choice(np.array([-1, 0, 1], dtype=np.int8), CN)
    on = route >= 0
    sb3 = [VecNormalizeReward(int(on.sum()), gamma, clip), VecNormalizeReward(int(on.sum()), gamma, clip)]
    dones = np.ones(int(on.sum()), dtype=bool)
    clipped = 0
    for it in range(6):
        rew = (rng.standard_normal((1, CN)) * (3.0 if it else 0.1) - 1.0).astype(np.float32)
        rew_d = np.minimum(rng.standard_normal(CN) * 4.0, 0.0).astype(np.float32)
        rms = merge(rms, batch_moments(rew, rew_d, route, gamma))
        got_c, got_d = scale(rew[0], rms[0][2], clip), scale(rew_d, rms[1][2], clip)
        want_c = sb3[0].step(rew[0, on].astype(np.float64), dones)
        want_d = sb3[1].step(rew_d[on].astype(np.float64), dones)
        np.testing.assert_allclose(got_c[on], want_c, rtol=1e-6, atol=0)
        np.testing.assert_allclose(got_d[on], want_d, rtol=1e-6, atol=0)
        assert _rel(rms[0][2], sb3[0].ret_rms.var) <= 1e-12 and _rel(rms[1][2], sb3[1].ret_rms.var) <= 1e-12
        clipped += int((np.abs(want_c) == clip).sum() + (np.abs(want_d) == clip).sum())
    if math.isfinite(clip) and clip < 1:
        assert clipped > 0                                   # the clip is exercised


def test_empty_batch_keeps_the_state():
    rms = np.array([[12.5, -3.0, 7.0], [3.0, -1.0, 0.25]])
    assert merge(rms, np.zeros(6)).tobytes() == rms.tobytes()
    rew, rew_d, route = _rollout(5, 40, 3, absent=1.0)
    mom = batch_moments(rew, rew_d, route, 0.99)
    assert (mom == 0).all() and merge(rms, mom).tobytes() == rms.tobytes()
    # one empty stream: only the other one moves
    mom = np.array([4.0, 2.0, 3.0, 0.0, 0.0, 0.0])
    out = merge(rms, mom)
    assert out[1].tobytes() == rms[1].tobytes() and out[0][0] == 16.5


def test_scale_rounds_once_and_does_not_subtract_the_mean():
    r = np.array([1.0, -1.0, 30.0, -30.0, 0.0], dtype=np.float32)
    got = scale(r, 3.0, 10.0)
    want = np.array([1 / math.sqrt(3.0 + 1e-8), -1 / math.sqrt(3.0 + 1e-8), 10.0, -10.0, 0.0], dtype=np.float32)
    assert got.tobytes() == want.tobytes()
    assert (scale(r, 3.0, math.inf)[2:4] == np.float32(np.array([30.0, -30.0]) / math.sqrt(3.0 + 1e-8))).all()
