"""Learning-rate schedules of Algo_PPO(lr_schedule="linear" | "adaptive") (DESIGN.md §4 "Learning-rate schedules"), no GPU: the
option checks of the constructor (which run before the env is touched), a float64 restatement of the adaptive rule at its
thresholds, NaN / inf and both clamp bounds, checked against rsl_rl's rule as written, the linear formula against CleanRL's
annealing, and an Adam whose lr changes every step against torch.optim.Adam.  tests/test_lr_schedule_gpu.py holds
mhppo_adam2_sched and the update to this restatement."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_grad_clip import clipped_adam64, _Untouchable  # noqa: E402

LR_MIN, LR_MAX = 1e-5, 1e-2


def adaptive_lr(lr, kl, delta):
    """One decision of the adaptive rule on an fp32 lr: the new fp32 lr, as a Python float.  kl > 2 delta divides by 1.5 (floor
    1e-5), 0 < kl < delta / 2 multiplies by 1.5 (ceiling 1e-2), anything else (NaN, +-inf included) keeps the lr; the change is
    computed in float64 and rounded to fp32."""
    lr = float(np.float32(lr))
    if math.isfinite(kl):
        if kl > 2.0 * delta:
            lr = float(np.float32(max(LR_MIN, lr / 1.5)))
        elif 0.0 < kl < 0.5 * delta:
            lr = float(np.float32(min(LR_MAX, lr * 1.5)))
    return lr


def linear_lr(lr0, k, K):
    """lr0 * max(0, 1 - k / K): the lr of the update after k completed iterations of a K-iteration anneal."""
    return lr0 * max(0.0, 1.0 - k / K)


def _rsl_rl(lr, kl, desired_kl):
    """rsl_rl's PPO.update, schedule == "adaptive", as written there (float64, no rounding)."""
    if kl > desired_kl * 2.0:
        lr = max(1e-5, lr / 1.5)
    elif kl < desired_kl / 2.0 and kl > 0.0:
        lr = min(1e-2, lr * 1.5)
    return lr


DELTA = 0.01
up, down = (lambda x: math.nextafter(x, math.inf)), (lambda x: math.nextafter(x, -math.inf))
KL_CASES = {  # kl -> expected direction: -1 divide, 0 keep, +1 multiply
    "2d": (2 * DELTA, 0), "2d+ulp": (up(2 * DELTA), -1), "2d-ulp": (down(2 * DELTA), 0),
    "d/2": (DELTA / 2, 0), "d/2-ulp": (down(DELTA / 2), 1), "d/2+ulp": (up(DELTA / 2), 0),
    "d": (DELTA, 0), "zero": (0.0, 0), "-zero": (-0.0, 0), "tiny": (5e-324, 1), "negative": (-1e-3, 0), "large": (1e30, -1),
    "nan": (math.nan, 0), "inf": (math.inf, 0), "-inf": (-math.inf, 0),
}


@pytest.mark.parametrize("case", list(KL_CASES))
def test_adaptive_rule_decisions(case):
    kl, direction = KL_CASES[case]
    lr = float(np.float32(3e-4))
    want = {-1: float(np.float32(lr / 1.5)), 0: lr, 1: float(np.float32(lr * 1.5))}[direction]
    assert adaptive_lr(lr, kl, DELTA) == want
    if math.isfinite(kl):                                           # rsl_rl's rule, rounded to fp32
        assert adaptive_lr(lr, kl, DELTA) == float(np.float32(_rsl_rl(lr, kl, DELTA)))
    else:                                                           # rsl_rl would divide at +inf; here a non-finite kl keeps the lr
        assert adaptive_lr(lr, kl, DELTA) == lr


@pytest.mark.parametrize("lr, kl, want", [
    (1e-5, 1.0, np.float32(1e-5)), (1.2e-5, 1.0, np.float32(1e-5)), (1.6e-5, 1.0, np.float32(1.6e-5 / 1.5)),
    (1e-2, 1e-4, np.float32(1e-2)), (8e-3, 1e-4, np.float32(1e-2)), (6e-3, 1e-4, np.float32(6e-3 * 1.5))])
def test_adaptive_rule_clamps(lr, kl, want):
    got = adaptive_lr(lr, kl, DELTA)
    assert got == float(want)
    assert got == float(np.float32(_rsl_rl(float(np.float32(lr)), kl, DELTA)))


def test_adaptive_rule_reaches_the_ceiling_from_the_default_actor_lr():
    """A pair whose KL stays below delta / 2 (the saturated choice actor) climbs from 3e-4 to the 1e-2 ceiling in 9 steps."""
    lr, steps = 3e-4, 0
    while lr < float(np.float32(LR_MAX)):
        lr, steps = adaptive_lr(lr, 1e-14, DELTA), steps + 1
    assert steps == 9 and lr == float(np.float32(LR_MAX))
    assert adaptive_lr(lr, 1e-14, DELTA) == lr


@pytest.mark.parametrize("k", [0, 1, 150, 299, 300, 301, 10 ** 6])
def test_linear_formula(k):
    K, lr0 = 300, 3e-4
    got = linear_lr(lr0, k, K)
    frac = 1.0 - ((k + 1) - 1.0) / K                               # CleanRL: iteration = k + 1, frac = 1 - (iteration - 1) / num_iterations
    assert got == (lr0 * frac if k < K else 0.0)
    assert got >= 0.0
    if k >= K:
        assert got == 0.0


def test_adam_with_a_new_lr_every_step_matches_torch():
    """The restated Adam step (tests/test_grad_clip.py, unclipped) with the lr changed before each step, against torch.optim.Adam
    with param_groups[0]["lr"] set before each step, float64."""
    g = torch.Generator().manual_seed(3)
    shapes = [(32, 13), (32,), (64, 32), (64,), (32, 64), (32,), (1, 32), (1,)]
    params = [torch.randn(s, generator=g, dtype=torch.float64, requires_grad=True) for s in shapes]
    flat = lambda ts: np.concatenate([t.detach().reshape(-1).numpy() for t in ts])
    p, m, v = flat(params), np.zeros(flat(params).size), np.zeros(flat(params).size)
    opt = torch.optim.Adam(params, lr=3e-4)
    lr = 3e-4
    for s, kl in enumerate([1e-3, 1e-3, 0.05, 0.01, 1e-4, 0.0, 0.03]):
        lr = adaptive_lr(lr, kl, DELTA)
        grads = [torch.randn(t.shape, generator=g, dtype=torch.float64) * 0.05 for t in params]
        for q, t in zip(params, grads):
            q.grad = t.clone()
        opt.param_groups[0]["lr"] = lr
        opt.step()
        p, m, v, _ = clipped_adam64(p, m, v, flat(grads), s + 1, lr, math.inf)
        np.testing.assert_allclose(flat(params), p, rtol=1e-13, atol=1e-15)


# ---------------------------------------------------------------------------------------------------------------------
# option checks

def _ctor(**opts):
    import mhppo_b200 as mh
    return mh.Algo_PPO(mh.Model_PPO, _Untouchable(), num_states_c=13, num_states_d=18, **opts)


BAD = {
    "unknown": dict(lr_schedule="cosine"), "upper": dict(lr_schedule="Linear"), "bool": dict(lr_schedule=True),
    "list": dict(lr_schedule=["linear"], lr_anneal_iterations=10),
    "adaptive_no_kl": dict(lr_schedule="adaptive"), "linear_no_K": dict(lr_schedule="linear"),
    "kl_without_adaptive": dict(desired_kl=0.01), "kl_with_linear": dict(lr_schedule="linear", lr_anneal_iterations=10, desired_kl=0.01),
    "K_without_linear": dict(lr_anneal_iterations=10), "K_with_adaptive": dict(lr_schedule="adaptive", desired_kl=0.01, lr_anneal_iterations=10),
}
for _i, _d in enumerate([True, False, math.nan, 0, 0.0, -0.01, math.inf, -math.inf, "0.01", np.bool_(True)]):
    BAD["desired_kl_%d" % _i] = dict(lr_schedule="adaptive", desired_kl=_d)
for _i, _k in enumerate([True, False, 0, -1, 300.0, 1.5, math.nan, math.inf, "300", np.float64(300)]):
    BAD["K_%d" % _i] = dict(lr_schedule="linear", lr_anneal_iterations=_k)


@pytest.mark.parametrize("case", list(BAD))
def test_lr_schedule_rejected_before_the_env_is_touched(case):
    with pytest.raises(ValueError):
        _ctor(**BAD[case])


@pytest.mark.parametrize("opts", [dict(lr_schedule=None), dict(lr_schedule="linear", lr_anneal_iterations=1),
                                  dict(lr_schedule="linear", lr_anneal_iterations=np.int64(300)),
                                  dict(lr_schedule="adaptive", desired_kl=0.01), dict(lr_schedule="adaptive", desired_kl=np.float32(0.02)),
                                  dict(lr_schedule="adaptive", desired_kl=1, target_kl=0.02, max_grad_norm=0.5)])
def test_lr_schedule_accepted(opts):
    """An accepted value passes the option checks: the constructor goes on to read the env."""
    with pytest.raises(AssertionError, match="touched the env"):
        _ctor(**opts)
