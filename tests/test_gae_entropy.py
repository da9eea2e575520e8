"""The two update options of Algo_PPO beyond the reference (DESIGN.md §4 "GAE and entropy options") restated in float64:
GAE(gamma, lambda) returns of the cross / wait buffers and the entropy bonus of the categorical choice actor.  The checks
here hold the restatements to their definitions and need no GPU; tests/test_gae_entropy_gpu.py holds the kernels
(mhppo_gae, mhppo_ppo_grad_ent) and Algo_PPO to these restatements.  The reference has neither option, so they live
here and not in oracle/."""
import numpy as np
import pytest
import torch

from oracle import ppo_oracle as PO


def gae_returns(rew, V, gamma, lam):
    """rew, V [T, ...] -> R [T, ...] in float64 with V(s_T) = 0 and R_T = 0:
    R_t = r_t + gamma * ((1 - lam) * V(s_{t+1}) + lam * R_{t+1}), in the operation order of k_gae (no contraction)."""
    rew, V = np.asarray(rew, np.float64), np.asarray(V, np.float64)
    R = np.zeros_like(rew)
    acc, vn = np.zeros(rew.shape[1:]), np.zeros(rew.shape[1:])
    for t in range(rew.shape[0] - 1, -1, -1):
        acc = rew[t] + gamma * ((1.0 - lam) * vn + lam * acc)
        R[t] = acc
        vn = V[t]
    return R


def gae_advantages_bruteforce(rew, V, gamma, lam):
    """The definition: A_t = sum_k (gamma lam)^k delta_{t+k}, delta_t = r_t + gamma V(s_{t+1}) - V(s_t), V(s_T) = 0."""
    rew, V = np.asarray(rew, np.float64), np.asarray(V, np.float64)
    T = rew.shape[0]
    Vn = np.concatenate([V[1:], np.zeros_like(V[:1])])
    delta = rew + gamma * Vn - V
    A = np.zeros_like(rew)
    for t in range(T):
        for k in range(T - t):
            A[t] += (gamma * lam) ** k * delta[t + k]
    return A


def _normalise(A):
    return (A - A.mean()) / (A.std() + 1e-10)                                    # PY:787 (unbiased std)


def choice_loss_ent(actor_sd, x, A, act, logp_old, c, n=None, dtype=torch.float64):
    """Loss and autograd gradients of the choice actor (train_model_d, PY:818-851, with the (M, M) broadcast in its f0 / f1
    closed form) plus the entropy bonus: loss = mean_s sum_k f_k surr_k(s) - c / n * sum_s H(pi(.|s)), H = -sum_k p_k log p_k.
    A: the advantages as the kernel sees them (rtg - V); n: the global sample count (default: the batch).  Returns
    (loss, {name: grad}, mean absolute per-sample term)."""
    x, A, act, logp_old = (torch.as_tensor(np.asarray(a), dtype=dtype) for a in (x, A, act, logp_old))
    n = x.shape[0] if n is None else n
    p = {k: v.detach().to(dtype).requires_grad_(True) for k, v in actor_sd.items()}
    h = torch.relu(x @ p["layer1.weight"].t() + p["layer1.bias"])
    h = torch.relu(h @ p["layer2.weight"].t() + p["layer2.bias"])
    h = torch.relu(h @ p["layer3.weight"].t() + p["layer3.bias"])
    z = (h @ p["layer4.weight"].t() + p["layer4.bias"])[:, :2]
    An = _normalise(A)
    logp = torch.log_softmax(z, dim=1)
    ratio = torch.exp(logp - logp_old[:, None])
    surr = -torch.min(ratio * An[:, None], torch.clamp(ratio, 0.8, 1.2) * An[:, None])
    f = torch.tensor([float((act == k).double().sum()) / n for k in (0, 1)], dtype=dtype)
    H = -(torch.exp(logp) * logp).sum(1)
    terms = (surr * f).sum(1) * (x.shape[0] / n) - c * H
    loss = terms.sum() / x.shape[0]
    grads = dict(zip(p, torch.autograd.grad(loss, list(p.values()))))
    return loss.item(), grads, float(terms.detach().abs().mean())


def entropy_dz(z, c, inv_n):
    """The kernel's closed form of the entropy term on logits z [M, 2]: H from log-softmax (z_k - m - log(e0 + e1)) and
    dLoss/dz_k = c * inv_n * p_k * (log p_k + H) of the loss term -c * inv_n * H."""
    z = np.asarray(z, np.float64)
    m = z.max(axis=1, keepdims=True)
    e = np.exp(z - m)
    lp = (z - m) - np.log(e.sum(axis=1, keepdims=True))
    p = e / e.sum(axis=1, keepdims=True)
    H = -(p * lp).sum(axis=1, keepdims=True)
    return -c * inv_n * H[:, 0], c * inv_n * p * (lp + H)


@pytest.mark.parametrize("T", [1, 2, 80])
@pytest.mark.parametrize("lam", [0.0, 0.5, 0.95, 1.0])
def test_lambda_return_equals_bruteforce_definition(T, lam):
    rng = np.random.default_rng(T * 10 + int(lam * 100))
    rew, V = rng.standard_normal((T, 7)) * 3 - 1, rng.standard_normal((T, 7)) * 5
    for gamma in (0.0, 0.99, 1.0):
        A = gae_returns(rew, V, gamma, lam) - V
        want = gae_advantages_bruteforce(rew, V, gamma, lam)
        np.testing.assert_allclose(A, want, rtol=0, atol=1e-12 * (1 + np.abs(rew).sum() + np.abs(V).sum()))


@pytest.mark.parametrize("T", [1, 2, 80])
def test_lambda_one_equals_reward_to_go_minus_value(T):
    """At lambda = 1 the restatement is the reference's estimator (futur_rewards, PY:658-684, gamma 0.99, zero bootstrap),
    bit for bit: the (1 - lambda) V term is an exact zero."""
    rng = np.random.default_rng(T)
    rew, V = rng.standard_normal((T, 5, 3)), rng.standard_normal((T, 5, 3)) * 4
    R = gae_returns(rew, V, 0.99, 1.0)
    assert np.array_equal(R, PO.reward_to_go(rew))
    assert np.array_equal(R - V, PO.reward_to_go(rew) - V)


def test_entropy_gradient_closed_form_equals_autograd():
    """The closed-form entropy gradient against float64 autograd of -c * inv_n * sum H, including logits 2000 apart (a
    saturated softmax: p = 0 exactly, yet the loss and the gradient stay finite)."""
    rng = np.random.default_rng(0)
    z = np.concatenate([rng.standard_normal((50, 2)) * 3, [[0.0, -2000.0], [1500.0, -500.0], [3.0, 2003.0], [7.0, 7.0]]])
    c, inv_n = 0.1, 1.0 / 37
    zt = torch.tensor(z, dtype=torch.float64, requires_grad=True)
    lp = torch.log_softmax(zt, dim=1)
    H = -(torch.exp(lp) * lp).sum(1)
    loss = -c * inv_n * H.sum()
    (g,) = torch.autograd.grad(loss, [zt])
    terms, dz = entropy_dz(z, c, inv_n)
    assert np.isfinite(dz).all() and np.isfinite(terms).all()
    np.testing.assert_allclose(terms.sum(), loss.item(), rtol=1e-13, atol=1e-300)
    np.testing.assert_allclose(dz, g.numpy(), rtol=1e-12, atol=1e-15)
    assert np.all(dz[50:52] == 0.0) and np.all(dz[52] == 0.0) and np.all(dz[53] == 0.0)   # saturated rows, and p = 1/2 exactly
