"""The update diagnostics of Algo_PPO(diagnostics=True) (DESIGN.md §4 "Diagnostics"), no GPU: float64 restatements of the four
diagnostics checked against their definitions, the host-side ratios of mhppo_b200.ppo.diag_ratios against them, and the
option checks of the constructor (which run before the env is touched).  tests/test_ppo_diagnostics_gpu.py holds the kernels
to these restatements."""
import math
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def k3(log_r):
    """r - 1 - log r, the k3 estimator of KL(old || new) per sample, as expm1(l) - l (no cancellation near r = 1)."""
    l = np.asarray(log_r, dtype=np.float64)
    return np.expm1(l) - l


def clipped(ratio):
    """1 where the clipped surrogate's clamp bites (r < 0.8 or r > 1.2), on the fp32 ratio the loss sees."""
    r = np.asarray(ratio, dtype=np.float32)
    return ((r < np.float32(0.8)) | (r > np.float32(1.2))).astype(np.float64)


def explained_variance(R, V):
    """1 - Var(R - V) / Var(R), population variances; NaN when Var(R) = 0."""
    R, V = np.asarray(R, np.float64), np.asarray(V, np.float64)
    vr = R.var()
    return 1.0 - (R - V).var() / vr if vr > 0 else float("nan")


def entropy2(z):
    """H of the two-way softmax of logits z [n, 2] in log-softmax form."""
    z = np.asarray(z, np.float64)
    lp = z - np.logaddexp(z[:, 0], z[:, 1])[:, None]
    return -(np.exp(lp) * lp).sum(1)


def record_sums(log_r, ratio, H, R, V):
    """The sums of one record row (include/mhppo.h, mhppo_ppo_grad_diag) from per-sample values, losses 0."""
    d = np.asarray(R, np.float64) - np.asarray(V, np.float64)
    R = np.asarray(R, np.float64)
    return [0.0, 0.0, k3(log_r).sum(), clipped(ratio).sum(), 0.0 if H is None else np.sum(H), d.sum(), (d * d).sum(), R.sum(), (R * R).sum()]


def test_k3_nonnegative_and_zero_at_one():
    l = np.concatenate([np.linspace(-700, 700, 20001), -np.logspace(-30, 2, 200), np.logspace(-30, 2, 200)])
    v = k3(l)
    assert np.isfinite(v).all() and (v >= 0).all()
    assert k3(0.0) == 0.0
    # second order near r = 1: l^2 / 2 (relative error of the expm1 form stays at the fp64 rounding level)
    small = np.array([1e-8, -1e-8, 1e-5, -1e-5])
    assert np.allclose(k3(small), small ** 2 / 2 + small ** 3 / 6, rtol=1e-6, atol=0)


def test_mean_k3_matches_gaussian_kl():
    """Samples a ~ N(mu0, s^2) of the old policy with r = p_new(a) / p_old(a), new = N(mu1, s^2): E[k3] = KL(old || new) =
    (mu0 - mu1)^2 / (2 s^2).  Bar: 6 standard errors of the sample mean of k3 (the estimator is unbiased)."""
    rng = np.random.default_rng(0)
    s = math.sqrt(0.5)
    for mu0, mu1 in ((0.0, 0.1), (-1.0, -0.7), (2.0, 2.5)):
        a = rng.normal(mu0, s, 2_000_000)
        log_r = (-(a - mu1) ** 2 + (a - mu0) ** 2) / (2 * s * s)
        v = k3(log_r)
        kl = (mu0 - mu1) ** 2 / (2 * s * s)
        se = v.std(ddof=1) / math.sqrt(len(v))
        assert abs(v.mean() - kl) <= 6 * se, (mu0, mu1, v.mean(), kl, se)


def test_explained_variance_definition():
    rng = np.random.default_rng(1)
    R = rng.normal(3.0, 2.0, 1000)
    assert explained_variance(R, R) == 1.0
    assert abs(explained_variance(R, np.full_like(R, R.mean()))) < 1e-12
    V = R + rng.normal(0, 1.0, 1000)
    assert explained_variance(R, V) < 1.0
    assert math.isnan(explained_variance(np.full(10, 4.0), np.zeros(10)))


def test_clip_fraction_boundaries():
    f = np.float32
    r = np.array([f(0.8), np.nextafter(f(0.8), f(0)), np.nextafter(f(0.8), f(2)), f(1.2), np.nextafter(f(1.2), f(2)),
                  np.nextafter(f(1.2), f(0)), f(1.0), f(0.0), f(np.inf)], dtype=np.float32)
    assert clipped(r).tolist() == [0, 1, 0, 0, 1, 0, 0, 1, 1]


def test_diag_ratios_restate_the_definitions():
    from mhppo_b200.ppo import diag_ratios
    rng = np.random.default_rng(2)
    n = 5000
    log_r = rng.normal(0, 0.2, n)
    ratio = np.exp(log_r).astype(np.float32)
    z = rng.normal(0, 2, (n, 2))
    R, V = rng.normal(-3, 5, n), rng.normal(-3, 4, n)
    H = entropy2(z)
    got = diag_ratios(record_sums(log_r, ratio, H, R, V), n, True)
    assert abs(got["approx_kl"] - k3(log_r).mean()) <= 1e-12 * k3(log_r).mean()
    assert got["clip_fraction"] == clipped(ratio).mean()
    assert abs(got["entropy"] - H.mean()) <= 1e-12
    assert abs(got["explained_variance"] - explained_variance(R, V)) <= 1e-10
    assert math.isnan(diag_ratios(record_sums(log_r, ratio, None, R, V), n, False)["entropy"])
    assert math.isnan(diag_ratios(record_sums(log_r, ratio, None, np.ones(n), V), n, False)["explained_variance"])


class _Untouchable:
    """An env stand-in that fails the test if the constructor reads anything from it."""
    def __getattr__(self, name):
        raise AssertionError("the constructor touched the env (%s) before checking its options" % name)


@pytest.mark.parametrize("opts", [dict(diagnostics=1), dict(diagnostics=None), dict(diagnostics="yes"), dict(diagnostics=np.bool_(True)),
                                  dict(target_kl=True), dict(target_kl=False), dict(target_kl=0), dict(target_kl=0.0), dict(target_kl=-0.01),
                                  dict(target_kl=math.inf), dict(target_kl=math.nan), dict(target_kl="0.01"), dict(target_kl=[0.01]),
                                  dict(diagnostics=False, target_kl=-1)])
def test_options_rejected_before_the_env_is_touched(opts):
    import mhppo_b200 as mh
    with pytest.raises(ValueError):
        mh.Algo_PPO(mh.Model_PPO, _Untouchable(), num_states_c=13, num_states_d=18, **opts)
