"""The PPO update kernels through the C ABI (mhppo_critic_grad_stats, mhppo_value_stats, mhppo_ppo_grad, mhppo_ppo_grad_dev,
mhppo_adam, mhppo_adam2) on synthetic sample buffers, against a float64 torch restatement of Algo_PPO.train_model_c /
train_model_d (PY:778-851) with autograd gradients.

The cases sit where the kernels can go wrong: sample counts at the tile and grid boundaries of every kernel (the grid is
read from the device), empty selections, dense (idx = NULL) and compacted sample lists, every input width up to 56,
clipped / unclipped / mixed surrogate batches, the ±1e3 placeholder features of absent cars, and Adam's bias correction
from step 1 to 10^6.  Inputs are redrawn until no hidden pre-activation and no ratio is a near-tie (see `_draw_batch`),
so fp32-versus-fp64 rounding is the only source of difference and the bars of DESIGN.md §4 apply unchanged:

    losses                     1e-5 of the mean absolute per-sample term (the loss itself unless the sum cancels)
    gradients                  1e-5 (exact-fp32 FFMA kernels) / 5e-5 (3xTF32 tensor-core kernels) of the largest entry
    V per element              rtol 1e-5, atol 1e-5
    advantage sums             1e-5 (FFMA) / 1e-4 (tensor cores), of sum |A| and of sum A^2

Exact properties: sample counts, the untouched (NaN) slots of V, zero gradient padding, empty selections, bitwise
repeatability of a launch, idx = NULL == idx = arange(CN), and a bitwise zero actor gradient for an all-clipped batch.
The two tests at the top check the reference itself and need no GPU."""
import math
import struct
import warnings

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as PO

BARS = {"loss": 1e-5, "grad_ffma": 1e-5, "grad_tc": 5e-5, "V": 1e-5, "stats_ffma": 1e-5, "stats_tc": 1e-4, "host_dev": 1e-6}
_WORST = {}          # largest measured error / bar per tolerance class (printed when the module ends)
LITERAL_MAX = 4096   # head 2: the literal (M, M) broadcast of PY:834-842 up to this many samples, the f0/f1 closed form above
DEFAULT_HEAD = (-1.0, 3.0, 0.5)
NAN_BITS = struct.unpack("<i", struct.pack("<f", float("nan")))[0]


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference of one epoch of train_model_c / train_model_d

def _net_sd(n_in, n_out, head, seed):
    torch.manual_seed(seed)
    return {k: v.detach().clone() for k, v in PO.Net(n_in, n_out, head).state_dict().items()}


def _mlp64(p, x):
    """Model_PPO's 4-layer MLP (PY:70-93) without the head; returns the raw outputs and the three hidden pre-activations."""
    z1 = x @ p["layer1.weight"].t() + p["layer1.bias"]
    z2 = torch.relu(z1) @ p["layer2.weight"].t() + p["layer2.bias"]
    z3 = torch.relu(z2) @ p["layer3.weight"].t() + p["layer3.bias"]
    return torch.relu(z3) @ p["layer4.weight"].t() + p["layer4.bias"], (z1, z2, z3)


def _leaf(sd, dtype=torch.float64):
    return {k: v.detach().to(dtype).requires_grad_(True) for k, v in sd.items()}


def _surrogate(ratio, adv):
    return -torch.min(ratio * adv, torch.clamp(ratio, 0.8, 1.2) * adv)          # PY:804-806


def reference_epoch(critic_sd, actor_sd, head, x, rtg, act, logp_old, gauss=DEFAULT_HEAD, literal=None, dtype=torch.float64):
    """Losses, gradients (autograd, float64) and intermediates of one epoch on the Q samples x [Q, D].  head 1: Gaussian
    actor (mu = tanh(z) * std + mean, a ~ N(mu, variance)); head 2: categorical choice actor, with the literal (M, M)
    broadcast of PY:834-842 when `literal` (default: Q <= LITERAL_MAX), else the f0 / f1 closed form.  dtype = float32
    gives what plain fp32 arithmetic achieves on the same batch (the yardstick of ill-conditioned batches)."""
    x, rtg, act, logp_old = (torch.as_tensor(np.asarray(a), dtype=dtype) for a in (x, rtg, act, logp_old))
    M = x.shape[0]
    pc, pa = _leaf(critic_sd, dtype), _leaf(actor_sd, dtype)
    out = {}
    Vo, out["pre_c"] = _mlp64(pc, x)
    V = Vo[:, 0]
    with torch.no_grad():                                                           # the magnitude the fp32 sums of V carry:
        m = x.abs()                                                                 # the critic on |x| with |W|, ReLU masks of x
        for l, z in zip((1, 2, 3), out["pre_c"]):
            m = (m @ pc["layer%d.weight" % l].abs().t() + pc["layer%d.bias" % l].abs()) * (z > 0)
        out["V_mag"] = (m @ pc["layer4.weight"].abs().t() + pc["layer4.bias"].abs())[:, 0].numpy()
    loss_c = torch.mean((V - rtg) ** 2)                                            # PY:808-809
    A = rtg - V.detach()                                                            # PY:786 (the actor loss does not reach the critic)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                                            # (the std of one sample is NaN, as in torch)
        An = (A - A.mean()) / (A.std() + 1e-10)                                     # PY:787
    o, out["pre_a"] = _mlp64(pa, x)
    if head == 1:
        mean, std, var = gauss
        mu = torch.tanh(o[:, 0]) * std + mean
        lp = -(act - mu) ** 2 / (2.0 * var) - 0.5 * math.log(2.0 * math.pi * var)   # MultivariateNormal(mu, var I).log_prob
        ratios = torch.exp(lp - logp_old)[:, None]
        terms = _surrogate(ratios[:, 0], An)
        loss_a = terms.mean()
        out["term_abs"] = float(terms.detach().abs().mean())
    else:
        literal = M <= LITERAL_MAX if literal is None else literal
        logp = torch.log_softmax(o[:, :2], dim=1)
        ratios = torch.exp(logp - logp_old[:, None])
        if literal:
            probs = torch.softmax(o[:, :2], dim=1)
            lpmm = torch.distributions.Categorical(probs).log_prob(act.reshape(-1, 1))       # (M, M): lp[i, j] = log p_j(a_i)
            terms = _surrogate(torch.exp(lpmm - logp_old), An)
            loss_a = terms.mean()
        else:
            f = torch.tensor([float((act == c).double().mean()) for c in (0, 1)], dtype=dtype)
            terms = torch.stack([_surrogate(ratios[:, c], An) for c in (0, 1)], dim=1)
            loss_a = (terms * f).sum(1).mean()
        out["term_abs"] = float(terms.detach().abs().mean()) if literal else float((terms.detach().abs() * f).sum(1).mean())
    out["grad_c"] = dict(zip(pc, torch.autograd.grad(loss_c, list(pc.values()))))
    ga = torch.autograd.grad(loss_a, list(pa.values()), allow_unused=True)
    out["grad_a"] = {k: (g if g is not None else torch.zeros_like(pa[k])) for k, g in zip(pa, ga)}
    out.update(loss_c=loss_c.item(), loss_a=loss_a.item(), V=V.detach().numpy(), A=A.numpy(), An=An.detach().numpy(),
               stats=(float(A.sum()), float((A * A).sum()), float(M)))
    return out


class _Grab:
    """Optimizer stand-in for oracle.ppo_oracle.train_step_*: keeps the gradients of its step() instead of stepping."""

    def __init__(self, params):
        self.params, self.grads = list(params), None

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    def step(self):
        self.grads = [p.grad.detach().clone() for p in self.params]


# ---------------------------------------------------------------------------------------------------------------------
# synthetic batches

def _preact_ties(pre):
    """Samples with a hidden pre-activation within 1e-3 of that layer's RMS of zero (the ReLU kink)."""
    bad = np.zeros(pre[0].shape[0], bool)
    for z in pre:
        z = z.detach().numpy()
        bad |= (np.abs(z) < 1e-3 * np.sqrt(np.mean(z * z))).any(axis=1)
    return bad


def _ratio_ties(r):
    return ((np.abs(r / 0.8 - 1) < 1e-3) | (np.abs(r / 1.2 - 1) < 1e-3)).any(axis=1)


def _draw_batch(rng, Q, D, head, critic_sd, actor_sd, regime="mixed", gauss=DEFAULT_HEAD, big_cols=False, actions=None):
    """Q samples (item order) of features, reward-to-go, action and old log-prob, fp32.  A drawn batch is evaluated in fp64
    and every sample with a near-tie is redrawn until none is left: a hidden pre-activation within 1e-3 of its layer's RMS
    of zero, a ratio within 1e-3 relative of 0.8 or 1.2, or a normalised advantage within 1e-3 of zero (its sign picks
    the clipped side).  regime: "mixed" ratios in [0.6, 1.4]; "noclip" every term on its unclipped branch; "clip" every
    term clipped (the actor gradient vanishes).  big_cols: every third feature column at ±1e3, like the x = -1000
    placeholder row of an absent car.  actions (head 2): "zeros" for a batch without action 1 (f1 = 0)."""
    def feats(n):
        x = rng.standard_normal((n, D)).astype(np.float32)
        if big_cols:
            x[:, ::3] = np.where(rng.random((n, len(range(0, D, 3)))) < 0.5, -1e3, 1e3)
        return x
    pc, pa = ({k: v.double() for k, v in sd.items()} for sd in (critic_sd, actor_sd))
    x = feats(Q)
    rtg = (rng.standard_normal(Q) * 5 - 3).astype(np.float32)
    for _ in range(200):
        x64 = torch.as_tensor(x, dtype=torch.float64)
        (V, pre_c), (o, pre_a) = _mlp64(pc, x64), _mlp64(pa, x64)
        bad = _preact_ties(pre_c) | _preact_ties(pre_a)
        if not bad.any():
            A = rtg - V[:, 0].numpy()
            An = (A - A.mean()) / (A.std(ddof=1) + 1e-10) if Q > 1 else np.ones(1)
            bad = np.abs(An) < 1e-3
            if not bad.any():
                break
            rtg[bad] = (rng.standard_normal(int(bad.sum())) * 5 - 3).astype(np.float32)
            continue
        x[bad] = feats(int(bad.sum()))
    else:
        raise AssertionError("could not draw a batch without near-ties")
    sign = np.where(An > 0, 1.0, -1.0)
    o = o.numpy()
    if head == 1:
        mean, std, var = gauss
        mu = np.tanh(o[:, 0]) * std + mean
        act = (mu + math.sqrt(var) * rng.standard_normal(Q)).astype(np.float32)
        lp_own = -(act.astype(np.float64) - mu) ** 2 / (2 * var) - 0.5 * math.log(2 * math.pi * var)
        lp_lo = lp_hi = lp_own
    else:
        lsm = o[:, :2] - np.logaddexp(o[:, 0], o[:, 1])[:, None]
        act = (np.zeros(Q) if actions == "zeros" else (rng.random(Q) >= np.exp(lsm[:, 0]))).astype(np.float32)   # a ~ the policy
        lp_own = np.where(act == 0, lsm[:, 0], lsm[:, 1])
        lp_lo, lp_hi = lsm.min(axis=1), lsm.max(axis=1)

    def old(idx):
        n = int(idx.sum())
        u = lambda a, b: rng.uniform(a, b, n)
        if regime == "mixed":
            return lp_own[idx] - np.log(u(0.6, 1.4))
        if regime == "noclip":       # advantage > 0: every ratio <= 1.2; < 0: every ratio >= 0.8
            return np.where(sign[idx] > 0, lp_hi[idx], lp_lo[idx]) - np.log(u(0.85, 1.15))
        assert regime == "clip"      # advantage > 0: every ratio > 1.2; < 0: every ratio < 0.8
        return np.where(sign[idx] > 0, lp_lo[idx] - np.log(u(1.3, 1.6)), lp_hi[idx] - np.log(u(0.5, 0.7)))
    logp = np.zeros(Q, np.float32)
    todo = np.ones(Q, bool)
    for _ in range(200):
        logp[todo] = old(todo).astype(np.float32)
        r = np.exp((np.stack([lp_own] if head == 1 else [lsm[:, 0], lsm[:, 1]], axis=1) - logp[:, None].astype(np.float64)))
        todo = _ratio_ties(r)
        if not todo.any():
            break
    else:
        raise AssertionError("could not draw ratios without near-ties")
    return dict(x=x, rtg=rtg, act=act, logp=logp)


# ---------------------------------------------------------------------------------------------------------------------
# checks of the reference itself (no GPU)

def test_reference_matches_oracle_autograd():
    """The fp64 reference against oracle.ppo_oracle (Net + train_step_c / train_step_d, fp32 autograd) on a small batch."""
    rng = np.random.default_rng(7)
    for head, D, n_out in ((1, 13, 1), (2, 30, 2)):
        csd, asd = _net_sd(D, 1, 0, 1), _net_sd(D, n_out, head, 2)
        b = _draw_batch(rng, 200, D, head, csd, asd)
        ref = reference_epoch(csd, asd, head, b["x"], b["rtg"], b["act"], b["logp"], literal=True)
        actor, critic = PO.Net(D, n_out, head), PO.Net(D, 1, 0)
        actor.load_state_dict(asd); critic.load_state_dict(csd)
        oa, oc = _Grab(actor.parameters()), _Grab(critic.parameters())
        step = PO.train_step_c if head == 1 else PO.train_step_d
        acts = b["act"][:, None] if head == 1 else b["act"].astype(np.int64)
        la, lc = step(actor, critic, oa, oc, b["x"], acts, b["logp"], b["rtg"])
        assert abs(la - ref["loss_a"]) <= 1e-5 * ref["term_abs"] and abs(lc - ref["loss_c"]) <= 1e-5 * ref["loss_c"]
        for grab, want in ((oa, ref["grad_a"]), (oc, ref["grad_c"])):
            scale = max(float(g.abs().max()) for g in want.values())
            for g, (k, w) in zip(grab.grads, want.items()):
                np.testing.assert_allclose(g.double().numpy(), w.numpy(), rtol=0, atol=2e-5 * scale, err_msg=k)


def test_reference_choice_closed_form_equals_literal_broadcast():
    """Head 2: the f0 / f1 closed form equals the literal (M, M) broadcast of PY:834-842 (mixed actions and all actions 0)."""
    rng = np.random.default_rng(3)
    csd, asd = _net_sd(18, 1, 0, 4), _net_sd(18, 2, 2, 5)
    for actions in (None, "zeros"):
        b = _draw_batch(rng, 300, 18, 2, csd, asd, actions=actions)
        lit = reference_epoch(csd, asd, 2, b["x"], b["rtg"], b["act"], b["logp"], literal=True)
        cf = reference_epoch(csd, asd, 2, b["x"], b["rtg"], b["act"], b["logp"], literal=False)
        assert abs(lit["loss_a"] - cf["loss_a"]) <= 1e-12 * lit["term_abs"]
        for k in lit["grad_a"]:
            np.testing.assert_allclose(cf["grad_a"][k].numpy(), lit["grad_a"][k].numpy(), rtol=1e-10, atol=1e-14, err_msg=k)


# ---------------------------------------------------------------------------------------------------------------------
# GPU side

def _L():
    import mhppo_b200
    return mhppo_b200.lib()


def _check(rc):
    from mhppo_b200._lib import check
    check(rc)


def _ptr(t):
    return None if t is None else t.data_ptr()


@pytest.fixture(params=[1, 2], ids=["ffma", "tc"])
def mode(request):
    """mhppo_set_mlp_mode 1 (exact-fp32 FFMA kernels) and 2 (tensor-core kernels wherever one exists; for the update,
    mode 0 takes the same kernels as mode 2)."""
    assert torch.cuda.is_available()
    L = _L()
    try:
        _check(L.mhppo_set_mlp_mode(request.param))
        yield request.param
        assert L.mhppo_tc_failures() == 0
    finally:
        L.mhppo_set_mlp_mode(0)
        L.mhppo_set_gaussian_head(*DEFAULT_HEAD, 2.0)


@pytest.fixture
def lib0():
    assert torch.cuda.is_available()
    L = _L()
    try:
        yield L
        assert L.mhppo_tc_failures() == 0
    finally:
        L.mhppo_set_mlp_mode(0)
        L.mhppo_set_gaussian_head(*DEFAULT_HEAD, 2.0)


@pytest.fixture(scope="module")
def ws():
    L = _L()
    return torch.zeros(max(L.mhppo_update_workspace_bytes(n) for n in (16, 32, 56)), dtype=torch.uint8, device="cuda")


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    if _WORST:
        print("\nlargest error / bar per tolerance class: " + ", ".join("%s %.3g" % kv for kv in sorted(_WORST.items())))


def _grid():
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    return min(sm, 148), min(2 * sm, 296)


def _record(cls, err, scale, bar):
    frac = float(err) / (bar * float(scale)) if scale > 0 else (0.0 if err == 0 else math.inf)
    _WORST[cls] = max(_WORST.get(cls, 0.0), frac)
    return frac


def _layout(T, K, CN, kind, rng):
    """Sample slots of the Q = T*K work items (item q -> t = q // K, k = q % K -> slot t*CN + idx[k]).  kind: "list" a
    shuffled compacted list of K of the CN columns, "arange" idx = arange(CN), "null" idx = NULL (K = CN), "empty" K = 0
    with the 1-element dummy list of Algo_PPO._selection."""
    if kind == "empty":
        idx, cols = np.zeros(1, np.int32), np.zeros(0, np.int64)
        K = 0
    elif kind == "list":
        cols = rng.permutation(CN)[:K]
        idx = cols.astype(np.int32)
    else:
        assert K == CN
        cols = np.arange(CN)
        idx = None if kind == "null" else cols.astype(np.int32)
    slots = (np.arange(T)[:, None] * CN + cols[None, :]).reshape(-1)
    return dict(T=T, K=K, CN=CN, S=T * CN, idx=None if idx is None else torch.as_tensor(idx, device="cuda"), slots=slots)


def _scatter(lay, v, rows=None):
    """Place the Q item values in their slots of an S-slot buffer; every other slot is NaN (a stray read poisons the result)."""
    S = lay["S"]
    if rows is None:
        out = np.full(S, np.nan, np.float32); out[lay["slots"]] = v
    else:
        out = np.full((rows, S), np.nan, np.float32); out[:, lay["slots"]] = v.T
    return torch.as_tensor(out, device="cuda")


def _pack(sd, n_in):
    from mhppo_b200.policy import _pack as pack
    return pack(sd, _L().mhppo_net_padded_in(n_in), "cpu")


def _bits_equal(a, b):
    return torch.equal(a.view(torch.int64 if a.dtype == torch.float64 else torch.int32), b.view(torch.int64 if b.dtype == torch.float64 else torch.int32))


def _uses_tc(mode, kp, D, head):
    return mode == 2 and kp == 16 and D <= 13 and head != 2


def run_case(mode, ws, lay, D, head, seed, regime="mixed", gauss=DEFAULT_HEAD, big_cols=False, actions=None, n_in=None):
    """One epoch of the update on the GPU (critic_grad_stats -> ppo_grad_dev, plus value_stats and the host-statistics
    ppo_grad) twice over, checked bit for bit between the two launches and against the fp64 reference."""
    L = _L()
    n_in = n_in or D
    kp = L.mhppo_net_padded_in(n_in)
    n_out = 2 if head == 2 else 1
    rng = np.random.default_rng(seed)
    csd, asd = _net_sd(n_in, 1, 0, seed), _net_sd(n_in, n_out, head, seed + 1)
    Q = lay["T"] * lay["K"]
    if gauss != DEFAULT_HEAD:
        _check(L.mhppo_set_gaussian_head(gauss[0], gauss[1], gauss[2], 2.0))
    b = _draw_batch(rng, max(Q, 1), D, head, csd, asd, regime, gauss, big_cols, actions) if Q else None
    if Q:
        x, rtg, act, logp = _scatter(lay, b["x"], D), _scatter(lay, b["rtg"]), _scatter(lay, b["act"]), _scatter(lay, b["logp"])
    else:
        x, rtg, act, logp = (torch.full(s, float("nan"), device="cuda") for s in ((D, lay["S"]), (lay["S"],), (lay["S"],), (lay["S"],)))
    net_c, net_a = _pack(csd, n_in).cuda(), _pack(asd, n_in).cuda()
    n_glob = Q if Q else 100            # an empty rank of a multi-GPU update still divides by the global count
    inv_n = 1.0 / n_glob
    f0 = float((b["act"] == 0).sum()) / n_glob if Q else 0.0
    f1 = float((b["act"] == 1).sum()) / n_glob if Q else 0.0
    npar = L.mhppo_net_param_count(n_in)
    idx, K, S, CN = lay["idx"], lay["K"], lay["S"], lay["CN"]

    def launch():
        o = {k: torch.full((S,), float("nan"), device="cuda") for k in ("V", "Vv")}
        o.update({k: torch.full((npar,), float("nan"), device="cuda") for k in ("gc", "ga", "gah")})
        o.update({k: torch.full((3,), float("nan"), dtype=torch.float64, device="cuda") for k in ("st", "stv")})
        o.update({k: torch.full((1,), float("nan"), dtype=torch.float64, device="cuda") for k in ("lc", "la", "lah")})
        _check(L.mhppo_critic_grad_stats(n_in, x.data_ptr(), D, S, _ptr(idx), K, CN, net_c.data_ptr(), rtg.data_ptr(), inv_n,
                                         o["gc"].data_ptr(), o["lc"].data_ptr(), o["V"].data_ptr(), o["st"].data_ptr(), ws.data_ptr(), None))
        _check(L.mhppo_value_stats(n_in, x.data_ptr(), D, S, _ptr(idx), K, CN, net_c.data_ptr(), rtg.data_ptr(), o["Vv"].data_ptr(),
                                   o["stv"].data_ptr(), ws.data_ptr(), None))
        _check(L.mhppo_ppo_grad_dev(n_in, head, x.data_ptr(), D, S, _ptr(idx), K, CN, net_a.data_ptr(), act.data_ptr(), logp.data_ptr(),
                                    rtg.data_ptr(), o["V"].data_ptr(), o["st"].data_ptr(), inv_n, f0, f1, o["ga"].data_ptr(),
                                    o["la"].data_ptr(), ws.data_ptr(), None))
        from mhppo_b200.ppo import combine_stats
        mean, inv_std, _ = combine_stats(o["st"].cpu())
        _check(L.mhppo_ppo_grad(n_in, head, x.data_ptr(), D, S, _ptr(idx), K, CN, net_a.data_ptr(), act.data_ptr(), logp.data_ptr(),
                                rtg.data_ptr(), o["V"].data_ptr(), mean, inv_std, inv_n, f0, f1, o["gah"].data_ptr(), o["lah"].data_ptr(),
                                ws.data_ptr(), None))
        torch.cuda.synchronize()
        return {k: v.cpu() for k, v in o.items()}

    o1, o2 = launch(), launch()
    fails = []

    def expect(ok, *what):
        if not ok:
            fails.append(what)
    for k in o1:                                               # fixed reduction order: bitwise repeatable
        expect(_bits_equal(o1[k], o2[k]), "not repeatable", k)
    o = o1
    # selected slots hold V, every other slot is still NaN bit for bit
    sel = np.zeros(S, bool); sel[lay["slots"]] = True
    for k in ("V", "Vv"):
        v = o[k].numpy()
        expect(np.isfinite(v[sel]).all(), "V not written", k)
        expect((o[k].view(torch.int32).numpy()[~sel] == NAN_BITS).all(), "V written outside the selection", k)
    expect(o["st"][2].item() == Q and o["stv"][2].item() == Q, "sample count", o["st"][2].item(), o["stv"][2].item(), Q)
    # padding of the flat gradient: W1t rows >= n_in, W4t columns >= n_out, b4 >= n_out
    for g in ("gc", "ga", "gah"):
        flat = o[g].numpy()
        no = 1 if g == "gc" else n_out
        w1 = flat[:kp * 32].reshape(kp, 32)
        w4 = flat[npar - 4 - 128:npar - 4].reshape(32, 4)
        expect((w1[n_in:] == 0).all() and (w4[:, no:] == 0).all() and (flat[npar - 4 + no:] == 0).all(), "padding", g)
    if Q == 0:
        for k in ("gc", "ga", "gah"):
            expect((o[k].view(torch.int32) == 0).all(), "empty selection: gradient", k)
        for k in ("lc", "la", "lah", "st", "stv"):
            expect((o[k] == 0).all(), "empty selection", k, o[k])
        assert not fails, fails
        return o
    # host statistics (Algo_PPO.combine_stats) vs statistics resolved in the kernel
    ga, gah = o["ga"].numpy().astype(np.float64), o["gah"].numpy().astype(np.float64)
    if Q == 1:
        # one sample: the unbiased std is NaN (torch gives the same), so is the actor loss; a NaN advantage takes neither branch
        # of the clipped surrogate, so the actor gradient is zero on both paths
        expect(math.isnan(o["la"].item()) and math.isnan(o["lah"].item()), "n = 1: actor loss", o["la"].item(), o["lah"].item())
        expect(np.array_equal(ga, gah) and (ga == 0).all(), "n = 1: actor gradient")
    else:
        # (not bit for bit: the kernel may contract sAA - n * mean^2 into an FMA)
        _record("host_dev", np.abs(ga - gah).max(), np.abs(ga).max(), BARS["host_dev"])
        expect(np.abs(ga - gah).max() <= BARS["host_dev"] * np.abs(ga).max(), "host vs device statistics: gradient")
    # against the fp64 reference
    ref = reference_epoch(csd, asd, head, b["x"], b["rtg"], b["act"], b["logp"], gauss)
    if Q > 1:
        expect(abs(o["la"].item() - o["lah"].item()) <= BARS["host_dev"] * ref["term_abs"], "host vs device statistics: loss")
    tc_c, tc_a = _uses_tc(mode, kp, D, 0), _uses_tc(mode, kp, D, head)
    tc_v = mode == 2 and kp == 16
    slots = lay["slots"]
    for k, tc in (("V", tc_c), ("Vv", tc_v)):
        got = o[k].numpy()[slots].astype(np.float64)
        tol = BARS["V"] * (1 + np.abs(ref["V"]))
        cls = "V"
        if big_cols:     # ±1e3 features: no fp32 evaluation reaches 1e-5 per element (DESIGN.md §4); bound by the magnitude of the sums
            tol = tol + (8 if tc else 1) * 2.0 ** -24 * ref["V_mag"]
            cls = "V_pm1e3_tc" if tc else "V_pm1e3_ffma"
        _record(cls, np.max(np.abs(got - ref["V"]) / tol), 1.0, 1.0)
        expect((np.abs(got - ref["V"]) <= tol).all(), "V", k, np.abs(got - ref["V"]).max())
    for k, tc in (("st", tc_c), ("stv", tc_v)):
        cls = "stats_tc" if tc else "stats_ffma"
        bar = BARS[cls]
        st = o[k].numpy()
        sA_abs = float(np.abs(ref["A"]).sum())
        _record(cls, abs(st[0] - ref["stats"][0]), sA_abs, bar)
        _record(cls, abs(st[1] - ref["stats"][1]), ref["stats"][1], bar)
        expect(abs(st[0] - ref["stats"][0]) <= bar * sA_abs, "sum A", k, st, ref["stats"])
        expect(abs(st[1] - ref["stats"][1]) <= bar * ref["stats"][1], "sum A^2", k, st, ref["stats"])
    lc = o["lc"].item()
    _record("loss", abs(lc - ref["loss_c"]), ref["loss_c"], BARS["loss"])
    expect(abs(lc - ref["loss_c"]) <= BARS["loss"] * ref["loss_c"], "critic loss", lc, ref["loss_c"])
    if Q > 1:
        la = o["la"].item()
        _record("loss", abs(la - ref["loss_a"]), ref["term_abs"], BARS["loss"])
        expect(abs(la - ref["loss_a"]) <= BARS["loss"] * ref["term_abs"], "actor loss", la, ref["loss_a"], ref["term_abs"])
    # ±1e3 features: the actor gradient is ill-conditioned in fp32 itself (DESIGN.md §4); the bar there is the larger of the usual
    # one and twice the error of plain fp32 autograd on the same batch
    ref32 = reference_epoch(csd, asd, head, b["x"], b["rtg"], b["act"], b["logp"], gauss, dtype=torch.float32) if big_cols else None
    for g, want_sd, tc in (("gc", ref["grad_c"], tc_c), ("ga", ref["grad_a"], tc_a)):
        if g == "ga" and Q == 1:
            continue
        want = _pack({k: v.detach() for k, v in want_sd.items()}, n_in).double().numpy()
        got = o[g].numpy().astype(np.float64)
        scale = np.abs(want).max()
        if regime == "clip" and g == "ga":
            expect(scale == 0.0 and (o[g].view(torch.int32) == 0).all(), "all-clipped batch: the actor gradient must be exactly zero")
            continue
        bar = BARS["grad_tc" if tc else "grad_ffma"]
        cls = "grad_tc" if tc else "grad_ffma"
        lim = bar * scale
        if big_cols:
            fp32 = _pack({k: v.detach() for k, v in ref32["grad_" + g[1]].items()}, n_in).double().numpy()
            lim = max(lim, 2 * np.abs(fp32 - want).max())
            cls += "_pm1e3"
            print("\n±1e3 %s head %d D %d mode %d: error / largest entry %.3g, fp32 autograd %.3g" % (
                g, head, D, mode, np.abs(got - want).max() / scale, np.abs(fp32 - want).max() / scale))
        _record(cls, np.abs(got - want).max(), lim, 1.0)
        expect(np.abs(got - want).max() <= lim, "gradient", g, np.abs(got - want).max() / scale, np.argmax(np.abs(got - want)))
    assert not fails, fails
    return o


# 1. tile and grid boundaries (n_in = 13, critic + Gaussian actor)
def _boundary_qs():
    G, V = _grid()
    return [0, 1, 127, 128, 129, 128 * G - 1, 128 * G, 128 * G + 1, 256 * G - 1, 256 * G, 256 * G + 1, 384 * G + 5, 256 * V + 1]


BOUNDARY_NAMES = ["0", "1", "127", "128", "129", "128G-1", "128G", "128G+1", "256G-1", "256G", "256G+1", "384G+5", "256V+1"]


@pytest.mark.gpu
@pytest.mark.parametrize("qi", range(len(BOUNDARY_NAMES)), ids=BOUNDARY_NAMES)
def test_tile_and_grid_boundaries(mode, ws, qi):
    """Sample counts that leave CTAs with 0, 1, 2 and 3+ tiles (and mixed counts in one launch) for the 128-sample tiles of
    k_ppo_grad_tc / k_value_stats_tc and the 256-sample tiles of k_ppo_grad<16> / k_value_stats<16>; Q = 0 is what a rank
    without routed samples runs in a multi-GPU update."""
    Q = _boundary_qs()[qi]
    rng = np.random.default_rng(100 + qi)
    lay = _layout(1, Q, Q + 7, "empty" if Q == 0 else "list", rng)
    run_case(mode, ws, lay, 13, 1, seed=10 + qi)


# 2. item -> sample mapping
@pytest.mark.gpu
def test_sample_mapping(mode, ws):
    """T > 1 with a shuffled compacted list, and the dense route (idx = NULL) against idx = arange(CN) bit for bit."""
    rng = np.random.default_rng(5)
    run_case(mode, ws, _layout(3, 43, 100, "list", rng), 13, 1, seed=20)
    CN = 61
    a = run_case(mode, ws, _layout(80, CN, CN, "null", rng), 13, 1, seed=21)
    b = run_case(mode, ws, _layout(80, CN, CN, "arange", rng), 13, 1, seed=21)
    for k in a:
        assert _bits_equal(a[k], b[k]), k


# 3. input widths
WIDTHS = [1, 12, 13, 14, 16, 17, 18, 30, 32, 33, 42, 54, 56]


@pytest.mark.gpu
@pytest.mark.parametrize("D", WIDTHS)
def test_input_widths(mode, ws, D):
    """Every padded width (16 / 32 / 56) at and around its edges, 12 = the older drivers' one-car choice width, 14-16 =
    16-padded inputs too wide for the tensor-core kernel's 13-feature staging: critic + choice actor at every width,
    critic + Gaussian actor up to 16.  Q = 256 G + 3 gives CTAs of 1, 2 and 3 tiles."""
    G, _ = _grid()
    rng = np.random.default_rng(D)
    Q = 256 * G + 3
    heads = (1, 2) if D <= 16 else (2,)
    for head in heads:
        run_case(mode, ws, _layout(1, Q, Q + 5, "list", rng), D, head, seed=1000 + 10 * D + head)


@pytest.mark.gpu
def test_input_width_rejections(lib0, ws):
    L = lib0
    x = torch.zeros(64 * 40, device="cuda")
    v = torch.zeros(40, device="cuda")
    g = torch.zeros(L.mhppo_net_param_count(56), device="cuda")
    st = torch.zeros(3, dtype=torch.float64, device="cuda")
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    idx = torch.arange(40, dtype=torch.int32, device="cuda")
    net = torch.zeros(L.mhppo_net_param_count(56), device="cuda")
    EINVAL, EUNSUP = -1, -5

    def calls(n_in, D, S, K, CN):
        p = x.data_ptr(), idx.data_ptr(), net.data_ptr(), v.data_ptr()
        return [L.mhppo_value_stats(n_in, p[0], D, S, p[1], K, CN, p[2], p[3], v.data_ptr(), st.data_ptr(), ws.data_ptr(), None),
                L.mhppo_critic_grad_stats(n_in, p[0], D, S, p[1], K, CN, p[2], p[3], 0.1, g.data_ptr(), loss.data_ptr(), v.data_ptr(),
                                          st.data_ptr(), ws.data_ptr(), None),
                L.mhppo_ppo_grad(n_in, 1, p[0], D, S, p[1], K, CN, p[2], p[3], p[3], p[3], p[3], 0.0, 1.0, 0.1, 0.0, 0.0, g.data_ptr(),
                                 loss.data_ptr(), ws.data_ptr(), None),
                L.mhppo_ppo_grad_dev(n_in, 2, p[0], D, S, p[1], K, CN, p[2], p[3], p[3], p[3], p[3], st.data_ptr(), 0.1, 0.5, 0.5,
                                     g.data_ptr(), loss.data_ptr(), ws.data_ptr(), None)]
    assert calls(57, 57, 40, 40, 40) == [EUNSUP] * 4
    assert L.mhppo_update_workspace_bytes(57) == -1 and L.mhppo_net_padded_in(57) == -1
    assert calls(13, 17, 40, 40, 40) == [EUNSUP] * 4          # D wider than the net's padded input
    assert calls(30, 33, 40, 40, 40) == [EUNSUP] * 4
    assert calls(13, 13, 40, 3, 30) == [EINVAL] * 4           # S not a multiple of CN
    assert calls(13, 13, 40, 21, 20) == [EINVAL] * 4          # K > CN
    torch.cuda.synchronize()


# 4. loss regimes, 5. feature scale
REGIMES = [(1, "mixed", DEFAULT_HEAD, None), (1, "clip", DEFAULT_HEAD, None), (1, "noclip", DEFAULT_HEAD, None),
           (1, "mixed", (-0.5, 2.5, 0.3), None), (1, "clip", (-0.5, 2.5, 0.3), None),
           (2, "mixed", DEFAULT_HEAD, None), (2, "clip", DEFAULT_HEAD, None), (2, "noclip", DEFAULT_HEAD, None),
           (2, "mixed", DEFAULT_HEAD, "zeros")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", REGIMES, ids=lambda c: "head%d-%s%s%s" % (c[0], c[1], "-gauss" if c[2] != DEFAULT_HEAD else "",
                                                                            "-actions0" if c[3] else ""))
def test_loss_regimes(mode, ws, case):
    """Clipped-surrogate branches of both actor heads: mixed, every term clipped (the actor gradient is exactly zero, the
    loss still matches), none clipped, a non-default Gaussian head, and a choice batch without action 1 (f1 = 0).
    Q = 3000 (the literal (M, M) reference)."""
    head, regime, gauss, actions = case
    rng = np.random.default_rng(REGIMES.index(case))
    D = 13 if head == 1 else 30
    run_case(mode, ws, _layout(3, 1000, 1100, "list", rng), D, head, seed=300 + REGIMES.index(case), regime=regime, gauss=gauss,
             actions=actions)


@pytest.mark.gpu
@pytest.mark.parametrize("head,D", [(1, 13), (2, 18), (2, 30)])
def test_placeholder_feature_scale(mode, ws, head, D):
    """A third of the feature columns at ±1e3, like the x = -1000 placeholder rows of absent cars that the choice nets and the
    tensor-core rollout see."""
    rng = np.random.default_rng(40 + D)
    G, _ = _grid()
    Q = 128 * G + 77
    run_case(mode, ws, _layout(2, Q // 2, Q // 2 + 9, "list", rng), D, head, seed=400 + D, big_cols=True)


# 7. Adam
B1, B2, EPS = 0.9, 0.999, 1e-8
f32 = lambda v: float(np.float32(v))


def _adam_ref(p, g, m, v, lr, step, scale=1.0):
    """One torch.optim.Adam step (PY:719-724) in fp64 from fp32 state, with the fp32 hyperparameters the C ABI receives.
    Returns p, m, v and the magnitudes the fp32 rounding of each result scales with."""
    b1, b2, eps, lr = f32(B1), f32(B2), f32(EPS), f32(lr)
    p, g, m, v = (np.asarray(a, np.float64) for a in (p, g, m, v))
    g = g * f32(scale)
    m1, v1 = b1 * m + (1 - b1) * g, b2 * v + (1 - b2) * g * g
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    ss = lr / bc1
    den = np.sqrt(v1) / math.sqrt(bc2) + eps
    p1 = p - ss * m1 / den
    m_mag, v_mag = np.abs(b1 * m) + np.abs((1 - b1) * g), np.abs(b2 * v) + (1 - b2) * g * g
    p_mag = np.abs(p) * 2 ** -22 + 2 ** -20 * ss * m_mag / den
    return p1, m1, v1, p_mag, m_mag * 2 ** -21, v_mag * 2 ** -21


def _adam_state(n, rng):
    p = rng.standard_normal(n).astype(np.float32)
    g = (rng.standard_normal(n) * 10.0 ** rng.uniform(-4, 1, n)).astype(np.float32)
    m = (rng.standard_normal(n) * 1e-2).astype(np.float32)
    v = (rng.random(n) * 1e-3).astype(np.float32)
    g[::5] = 0; v[::7] = 0; m[::35] = 0           # g = 0, v = 0, and entries with m = v = g = 0 (p must not move)
    return p, g, m, v


def _check_adam(got, want, tag):
    for name, a, w, tol in zip("pmv", got, want[:3], want[3:]):
        a = a.cpu().numpy().astype(np.float64)
        err = np.abs(a - w)
        _record("adam_step", np.max(err / np.maximum(tol, 1e-45)), 1.0, 1.0)
        assert (err <= tol).all(), (tag, name, int(np.argmax(err - tol)), err.max())


ADAM_N = [1, 255, 256, 257, 4868, 5380]
ADAM_STEPS = [1, 2, 10, 1000, 10 ** 6]


@pytest.mark.gpu
@pytest.mark.parametrize("step", ADAM_STEPS)
def test_adam_single_step(lib0, step):
    """mhppo_adam (grad_scale != 1) against one torch.optim.Adam step in fp64, every size around the 256-thread blocks and the
    flat sizes of the 16- and 32-padded nets.  The tolerance is a few fp32 roundings of each result's terms."""
    L = lib0
    rng = np.random.default_rng(step)
    for n in ADAM_N:
        p, g, m, v = _adam_state(n, rng)
        t = [torch.as_tensor(a.copy(), device="cuda") for a in (p, g, m, v)]
        _check(L.mhppo_adam(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), n, 3e-4, B1, B2, EPS, step, 0.37, None))
        torch.cuda.synchronize()
        _check_adam((t[0], t[2], t[3]), _adam_ref(p, g, m, v, 3e-4, step, 0.37), ("adam", n, step))
        assert np.array_equal(t[0].cpu().numpy()[::35], p[::35])


@pytest.mark.gpu
@pytest.mark.parametrize("step", ADAM_STEPS)
def test_adam2_single_step(lib0, step):
    """mhppo_adam2: both nets of a pair in one launch, with n0 != n1 both ways, lr0 != lr1 and step0 != step1."""
    L = lib0
    rng = np.random.default_rng(50 + step)
    step1 = step + 1 if step < 10 else step // 2 + 1
    for n0, n1 in ((1, 5380), (5380, 1), (255, 257), (257, 255), (4868, 5380), (5380, 4868), (256, 256)):
        s0, s1 = _adam_state(n0, rng), _adam_state(n1, rng)
        t0 = [torch.as_tensor(a.copy(), device="cuda") for a in s0]
        t1 = [torch.as_tensor(a.copy(), device="cuda") for a in s1]
        _check(L.mhppo_adam2(t0[0].data_ptr(), t0[1].data_ptr(), t0[2].data_ptr(), t0[3].data_ptr(), n0, 3e-4, step,
                             t1[0].data_ptr(), t1[1].data_ptr(), t1[2].data_ptr(), t1[3].data_ptr(), n1, 1e-3, step1, B1, B2, EPS, None))
        torch.cuda.synchronize()
        _check_adam((t0[0], t0[2], t0[3]), _adam_ref(*s0, 3e-4, step), ("adam2 net0", n0, n1, step))
        _check_adam((t1[0], t1[2], t1[3]), _adam_ref(*s1, 1e-3, step1), ("adam2 net1", n0, n1, step1))


@pytest.mark.gpu
def test_adam_trajectory_matches_torch(lib0):
    """1000 steps of mhppo_adam and of both halves of mhppo_adam2 against torch.optim.Adam in fp32 on the CPU, on the same
    gradient sequence (magnitudes 1e-6 .. 1e2, every 7th entry always zero).  Bound: |p - p_torch| <= 1e-5 * sum_t |dp_t|
    (the path length of the entry) + 2^-22 |p|; the two fp32 implementations round differently (lerp vs multiply-add,
    division vs reciprocal) but neither error compounds."""
    L = lib0
    rng = np.random.default_rng(11)
    n0, n1, T = 4868, 5380, 1000
    nets = []
    for n, lr in ((n0, 3e-4), (n1, 1e-3), (n0, 3e-4)):
        p = rng.standard_normal(n).astype(np.float32)
        tp = torch.tensor(p.copy(), requires_grad=True)
        nets.append(dict(n=n, lr=lr, dev=[torch.as_tensor(p.copy(), device="cuda")] + [torch.zeros(n, device="cuda") for _ in range(2)],
                         tp=tp, opt=torch.optim.Adam([tp], lr=lr), path=np.zeros(n)))
    for t in range(1, T + 1):
        gs = []
        for net in nets:
            g = (rng.standard_normal(net["n"]) * 10.0 ** rng.uniform(-6, 2)).astype(np.float32)
            g[::7] = 0
            gs.append(torch.as_tensor(g, device="cuda"))
            before = net["tp"].detach().clone()
            net["tp"].grad = torch.as_tensor(g)
            net["opt"].step()
            net["path"] += np.abs((net["tp"].detach() - before).numpy())
        a, b, c = nets
        _check(L.mhppo_adam2(a["dev"][0].data_ptr(), gs[0].data_ptr(), a["dev"][1].data_ptr(), a["dev"][2].data_ptr(), n0, a["lr"], t,
                             b["dev"][0].data_ptr(), gs[1].data_ptr(), b["dev"][1].data_ptr(), b["dev"][2].data_ptr(), n1, b["lr"], t,
                             B1, B2, EPS, None))
        _check(L.mhppo_adam(c["dev"][0].data_ptr(), gs[2].data_ptr(), c["dev"][1].data_ptr(), c["dev"][2].data_ptr(), n0, c["lr"],
                            B1, B2, EPS, t, 1.0, None))
    torch.cuda.synchronize()
    for net in nets:
        got, want = net["dev"][0].cpu().numpy().astype(np.float64), net["tp"].detach().numpy().astype(np.float64)
        tol = 1e-5 * net["path"] + 2 ** -22 * np.abs(want)
        _record("adam_trajectory", np.max(np.abs(got - want) / tol), 1.0, 1.0)
        assert (np.abs(got - want) <= tol).all(), np.max(np.abs(got - want) / tol)


@pytest.mark.gpu
def test_adam_rejects_invalid_arguments(lib0):
    L = lib0
    t = torch.zeros(8, device="cuda")
    q = t.data_ptr()
    for n, step in ((0, 1), (-3, 1), (8, 0), (8, -1)):
        assert L.mhppo_adam(q, q, q, q, n, 1e-3, B1, B2, EPS, step, 1.0, None) == -1
    for n0, n1, s0, s1 in ((0, 8, 1, 1), (8, 0, 1, 1), (8, 8, 0, 1), (8, 8, 1, 0), (-1, 8, 1, 1)):
        assert L.mhppo_adam2(q, q, q, q, n0, 1e-3, s0, q, q, q, q, n1, 1e-3, s1, B1, B2, EPS, None) == -1
    assert torch.equal(t.cpu(), torch.zeros(8))
