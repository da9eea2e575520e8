"""Per-net gradient-norm clipping of Algo_PPO(max_grad_norm=g) (DESIGN.md §5 "Gradient-norm clipping"), no GPU: the option checks
of the constructor (which run before the env is touched), and a float64 restatement of the clip rule and of the clipped Adam step,
checked against torch.nn.utils.clip_grad_norm_ on CPU tensors.  tests/test_grad_clip_gpu.py holds mhppo_adam2_clip and the update
to this restatement."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def clip_coef(norm, max_norm):
    """torch's factor max_norm / (norm + 1e-6), applied only when it is < 1; a non-finite norm leaves the gradient unchanged."""
    if not math.isfinite(norm):
        return 1.0
    c = max_norm / (norm + 1e-6)
    return c if c < 1.0 else 1.0


def clipped_adam64(p, m, v, g, step, lr, max_norm, beta1=0.9, beta2=0.999, eps=1e-8):
    """One net's clipped Adam step in float64 (torch.optim.Adam defaults after clip_grad_norm_): returns (p, m, v, norm)."""
    p, m, v, g = (np.asarray(a, np.float64) for a in (p, m, v, g))
    norm = math.sqrt(float(np.dot(g, g)))
    gi = g * clip_coef(norm, max_norm)
    m = beta1 * m + (1.0 - beta1) * gi
    v = beta2 * v + (1.0 - beta2) * gi * gi
    bc1, bc2 = 1.0 - beta1 ** step, 1.0 - beta2 ** step
    return p - (lr / bc1) * (m / (np.sqrt(v) / math.sqrt(bc2) + eps)), m, v, norm


def _ref_grads(seed, scale, n_in=13, n_out=1):
    """The gradient of one net in the reference layout (the state_dict tensors of Model_PPO), float64."""
    g = torch.Generator().manual_seed(seed)
    shapes = [(32, n_in), (32,), (64, 32), (64,), (32, 64), (32,), (n_out, 32), (n_out,)]
    return [torch.randn(s, generator=g, dtype=torch.float64) * scale for s in shapes]


def _torch_clip(grads, max_norm):
    params = [torch.zeros_like(t, requires_grad=True) for t in grads]
    for q, t in zip(params, grads):
        q.grad = t.clone()
    total = torch.nn.utils.clip_grad_norm_(params, max_norm)
    return float(total), [q.grad for q in params]


@pytest.mark.parametrize("case", ["below", "above", "at", "zero", "inf"])
def test_clip_rule_matches_torch(case):
    grads = _ref_grads(1, 0.0 if case == "zero" else 0.05)
    flat = torch.cat([t.reshape(-1) for t in grads]).numpy()
    norm = math.sqrt(float(np.dot(flat, flat)))
    max_norm = {"below": 10.0 * norm, "above": 0.1 * norm, "at": norm, "zero": 0.5, "inf": math.inf}[case]
    t_norm, t_grads = _torch_clip(grads, max_norm)
    assert abs(t_norm - norm) <= 1e-12 * max(norm, 1e-300)
    coef = clip_coef(norm, max_norm)
    if case in ("below", "zero", "inf"):
        assert coef == 1.0
    else:
        assert coef < 1.0                     # at the threshold the 1e-6 of the denominator still scales by norm / (norm + 1e-6)
    for a, b in zip(t_grads, grads):
        assert torch.allclose(a, b * coef, rtol=1e-14, atol=0.0)


@pytest.mark.parametrize("bad", [math.inf, math.nan])
def test_non_finite_norm_leaves_the_step_unclipped(bad):
    """torch reports the same non-finite norm, but would multiply the gradient by 0 (inf) or NaN; the option instead takes the
    unclipped step, so clipping adds no failure mode of its own."""
    grads = _ref_grads(2, 0.05)
    grads[3][5] = bad
    flat = torch.cat([t.reshape(-1) for t in grads]).numpy()
    norm = math.sqrt(float(np.dot(flat, flat)))
    t_norm, _ = _torch_clip(grads, 0.5)
    assert math.isinf(norm) == math.isinf(t_norm) and math.isnan(norm) == math.isnan(t_norm)
    assert clip_coef(norm, 0.5) == 1.0
    rng = np.random.default_rng(0)
    p, m, v = rng.normal(size=flat.size), rng.normal(size=flat.size) * 1e-3, rng.random(flat.size) * 1e-6
    with np.errstate(invalid="ignore"):                                    # inf / inf in the step of the inf element
        a = clipped_adam64(p, m, v, flat, 3, 1e-3, 0.5)
        b = clipped_adam64(p, m, v, flat, 3, 1e-3, math.inf)
    for x, y in zip(a[:3], b[:3]):
        np.testing.assert_array_equal(x, y)


def test_clipped_adam_matches_torch_optimiser():
    """The restated step against torch.optim.Adam after clip_grad_norm_, over three steps that clip."""
    grads = [_ref_grads(10 + s, 0.05) for s in range(3)]
    params = [torch.randn(t.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(7 + i), requires_grad=True)
              for i, t in enumerate(grads[0])]
    flat = lambda ts: np.concatenate([t.detach().reshape(-1).numpy() for t in ts])
    p, m, v = flat(params), np.zeros(flat(params).size), np.zeros(flat(params).size)
    opt = torch.optim.Adam(params, lr=3e-4)
    for s, gs in enumerate(grads):
        for q, t in zip(params, gs):
            q.grad = t.clone()
        torch.nn.utils.clip_grad_norm_(params, 0.2)
        opt.step()
        p, m, v, norm = clipped_adam64(p, m, v, flat(gs), s + 1, 3e-4, 0.2)
        assert clip_coef(norm, 0.2) < 1.0
        np.testing.assert_allclose(flat(params), p, rtol=1e-13, atol=1e-15)


def test_norm_over_the_flat_layout_is_the_reference_norm():
    """The flat kernel layout pads W1^T to KP rows and layer 4 to 4 outputs; with those slots 0 (as the gradient passes leave them)
    the norm over the flat buffer equals the norm over the reference-layout tensors."""
    from mhppo_b200.policy import _pack
    for n_in, kp, n_out in ((13, 16, 1), (18, 32, 2), (30, 32, 2), (54, 56, 2)):
        grads = _ref_grads(n_in, 0.05, n_in, n_out)
        sd = dict(zip(["layer%d.%s" % (i // 2 + 1, "weight" if i % 2 == 0 else "bias") for i in range(8)], grads))
        f = _pack(sd, kp, "cpu").double().numpy()
        ref = torch.cat([t.reshape(-1) for t in grads]).float().double().numpy()
        assert f.size - ref.size == (kp - n_in) * 32 + 33 * (4 - n_out)
        nf, nr = math.sqrt(float(np.dot(f, f))), math.sqrt(float(np.dot(ref, ref)))
        assert abs(nf - nr) <= 1e-14 * nr


class _Untouchable:
    """An env stand-in that fails the test if the constructor reads anything from it."""
    def __getattr__(self, name):
        raise AssertionError("the constructor touched the env (%s) before checking its options" % name)


@pytest.mark.parametrize("bad", [True, False, math.nan, 0, 0.0, -0.5, -math.inf, "0.5", [0.5], np.bool_(True), complex(0.5, 0)])
def test_max_grad_norm_rejected_before_the_env_is_touched(bad):
    import mhppo_b200 as mh
    with pytest.raises(ValueError):
        mh.Algo_PPO(mh.Model_PPO, _Untouchable(), num_states_c=13, num_states_d=18, max_grad_norm=bad)


@pytest.mark.parametrize("good", [None, 0.5, 1, math.inf, np.float32(0.5)])
def test_max_grad_norm_accepted(good):
    """An accepted value passes the option checks: the constructor goes on to read the env."""
    import mhppo_b200 as mh
    with pytest.raises(AssertionError, match="touched the env"):
        mh.Algo_PPO(mh.Model_PPO, _Untouchable(), num_states_c=13, num_states_d=18, max_grad_norm=good)
