"""The GAE and entropy options of the update on the GPU: mhppo_gae and mhppo_ppo_grad_ent through the C ABI, and
Algo_PPO(gae_lambda=..., entropy_coef=...) on real rollouts, against the float64 restatements of tests/test_gae_entropy.py.

Bars (DESIGN.md §4): ret within 1 fp32 ulp of the fp64 recursion, advantage sums 1e-9 of sum |A| / relative, counts exact;
losses 1e-5 relative (of the mean absolute per-sample term for the actor), gradients 1e-5 (FFMA) / 5e-5 (3xTF32) of the
largest entry, weights after a 10-epoch update 1e-4 (FFMA) / 2.5e-4 (3xTF32) of the largest weight.  The PPO-level cases run in the three
mhppo_set_mlp_mode modes.  Run as a script under torch.distributed.run it is the two-rank check of the options."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_gae_entropy import choice_loss_ent, gae_returns  # noqa: E402
from test_update_kernels_gpu import _draw_batch, _grid, _mlp64, _net_sd, _pack, _bits_equal  # noqa: E402

pytestmark = pytest.mark.gpu
EINVAL = -1


def _lib():
    import mhppo_b200
    return mhppo_b200.lib()


def _check(rc):
    from mhppo_b200._lib import check
    check(rc)


@pytest.fixture
def lib0():
    assert torch.cuda.is_available()
    L = _lib()
    try:
        yield L
        assert L.mhppo_tc_failures() == 0
    finally:
        L.mhppo_set_mlp_mode(0)


@pytest.fixture(params=[0, 1, 2], ids=["auto", "ffma", "tc"])
def mlp_mode(request):
    assert torch.cuda.is_available()
    L = _lib()
    try:
        _check(L.mhppo_set_mlp_mode(request.param))
        yield request.param
        assert L.mhppo_tc_failures() == 0
    finally:
        L.mhppo_set_mlp_mode(0)


@pytest.fixture(scope="module")
def ws():
    L = _lib()                                           # the largest update workspace (56-padded nets) serves every call
    return torch.zeros(max(L.mhppo_update_workspace_bytes(n) for n in (13, 32, 56)), dtype=torch.uint8, device="cuda")


# ---------------------------------------------------------------------------------------------------------------------
# 1. mhppo_gae against the fp64 recursion

def _gae_inputs(T, CN, seed):
    rng = np.random.default_rng(seed)
    route = rng.choice(np.array([-1, 0, 1], np.int8), CN, p=[0.2, 0.4, 0.4])
    route[:min(CN, 3)] = [-1, 0, 1][:min(CN, 3)] if CN > 1 else [0]
    rew = (rng.standard_normal((T, CN)) * 2 - 1).astype(np.float32)
    V = (rng.standard_normal((T, CN)) * 5).astype(np.float32)
    V[:, route < 0] = np.nan                             # absent columns must not be read
    return route, rew, V


def _run_gae(L, ws, rew_d, V_d, route_d, T, CN, gamma, lam):
    ret = torch.full((T * CN,), float("nan"), device="cuda")
    st = torch.full((6,), float("nan"), dtype=torch.float64, device="cuda")
    _check(L.mhppo_gae(rew_d.data_ptr(), V_d.data_ptr(), route_d.data_ptr(), T, CN, gamma, lam, ret.data_ptr(), st.data_ptr(),
                       ws.data_ptr(), None))
    return ret, st


@pytest.mark.parametrize("CN", [1, 255, 256, 257, 524288])
@pytest.mark.parametrize("T", [1, 2, 80])
def test_gae_kernel_matches_fp64(lib0, ws, T, CN):
    L = lib0
    route, rew, V = _gae_inputs(T, CN, 7 * T + CN)
    rew_d, V_d, route_d = (torch.as_tensor(a.reshape(-1), device="cuda") for a in (rew, V, route))
    present = route >= 0
    for gamma in (0.0, 0.99, 1.0):
        for lam in (0.0, 0.5, 0.95, 1.0):
            r1, s1 = _run_gae(L, ws, rew_d, V_d, route_d, T, CN, gamma, lam)
            r2, s2 = _run_gae(L, ws, rew_d, V_d, route_d, T, CN, gamma, lam)
            assert _bits_equal(r1, r2) and _bits_equal(s1, s2), ("not repeatable", gamma, lam)
            ret, st = r1.cpu().numpy().reshape(T, CN), s1.cpu().numpy()
            assert (ret[:, ~present].view(np.int32) == 0).all(), "absent columns must be written +0"
            R = gae_returns(rew[:, present], V[:, present], gamma, lam)
            got = ret[:, present].astype(np.float64)
            ulp = np.spacing(np.abs(R).astype(np.float32)).astype(np.float64)
            assert (np.abs(got - R) <= ulp).all(), ("ret", gamma, lam, np.max(np.abs(got - R) / ulp))
            A = (R.astype(np.float32) - V[:, present]).astype(np.float64)      # the advantage as the actor forms it, fp32
            rsel = route[present]
            for r in (0, 1):
                a = A[:, rsel == r]
                sA, sAA, n = st[3 * r:3 * r + 3]
                assert n == a.size, ("count", r, n, a.size)
                assert abs(sA - a.sum()) <= 1e-9 * np.abs(a).sum(), ("sum A", r, sA, a.sum())
                assert abs(sAA - (a * a).sum()) <= 1e-9 * (a * a).sum(), ("sum A^2", r, sAA, (a * a).sum())


def test_gae_rejects_invalid_arguments(lib0, ws):
    L = lib0
    T, CN = 4, 10
    f = torch.zeros(T * CN, device="cuda")
    route = torch.zeros(CN, dtype=torch.int8, device="cuda")
    st = torch.zeros(6, dtype=torch.float64, device="cuda")
    p = dict(rew=f.data_ptr(), V=f.data_ptr(), route=route.data_ptr(), ret=f.data_ptr(), st=st.data_ptr(), ws=ws.data_ptr())

    def call(T=T, CN=CN, gamma=0.99, lam=0.95, **null):
        q = {k: (None if null.get(k) else v) for k, v in p.items()}
        return L.mhppo_gae(q["rew"], q["V"], q["route"], T, CN, gamma, lam, q["ret"], q["st"], q["ws"], None)
    for k in p:
        assert call(**{k: True}) == EINVAL, k
    for bad in (dict(T=0), dict(T=-1), dict(CN=0), dict(CN=-5), dict(gamma=-1e-9), dict(gamma=1.0 + 1e-12), dict(gamma=math.nan),
                dict(gamma=math.inf), dict(lam=-0.5), dict(lam=1.5), dict(lam=math.nan), dict(lam=-math.inf)):
        assert call(**bad) == EINVAL, bad
    assert call(gamma=0.0, lam=0.0) == 0 and call(gamma=1.0, lam=1.0) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 2. lambda = 1 is the existing path

@pytest.mark.parametrize("T,CN", [(1, 257), (80, 1000), (80, 524288)])
def test_gae_lambda_one_equals_returns_bitwise(lib0, ws, T, CN):
    L = lib0
    route, rew, V = _gae_inputs(T, CN, T + CN)
    rew_d, V_d, route_d = (torch.as_tensor(a.reshape(-1), device="cuda") for a in (rew, V, route))
    rl = torch.zeros(T * CN, device="cuda")
    rtg, rew_dd = torch.zeros(T * CN, device="cuda"), torch.zeros(CN, device="cuda")
    _check(L.mhppo_returns(rew_d.data_ptr(), rl.data_ptr(), T, CN, 0.99, rtg.data_ptr(), rew_dd.data_ptr(), None))
    ret, _ = _run_gae(L, ws, rew_d, V_d, route_d, T, CN, 0.99, 1.0)
    present = torch.as_tensor(route >= 0, device="cuda")
    assert _bits_equal(ret.view(T, CN)[:, present].contiguous(), rtg.view(T, CN)[:, present].contiguous())


def _algo(N, seed=3, nb=(4, 3, 2), **opts):
    import mhppo_b200 as mh
    nb_car, nb_ped, nb_lines = nb
    env = mh.VecCrosswalkEnv("coop_scalable", N, nb_car=nb_car, nb_ped=nb_ped, nb_lines=nb_lines, seed=seed, env_id0=0)
    torch.manual_seed(0)
    D = 2 + 6 * (2 * nb_lines - 1) + 10
    algo = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=D, num_actions=1, mean=-1.0, std=3.0, nb_cars=nb_car, dt=0.3,
                       **opts)
    algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
    return algo


def _grad_bar(mode):
    return 5e-5 if mode in (0, 2) else 1e-5           # the 13-input update runs on the tensor cores in modes auto and tc


def test_gae_lambda_one_first_epoch_matches_reference_mode(mlp_mode):
    """GAE mode at lambda = 1 (V_old from mhppo_value_stats, targets from mhppo_gae) against reference mode (V from
    mhppo_critic_grad_stats, targets from mhppo_returns) on the same rollout: the first epoch's gradients agree at the bars;
    the choice pair, which GAE mode leaves alone, is bit-identical."""
    ref, gae = _algo(2048), _algo(2048, gae_lambda=1.0)
    for name in ("act", "logp", "rew", "rtg", "obs_c"):
        assert torch.equal(getattr(ref.rollout, name), getattr(gae.rollout, name)), name
    ref.update(epochs=1)
    gae.update(epochs=1)
    torch.cuda.synchronize()
    assert _bits_equal(gae.rollout.ret.view(-1)[gae.rollout.route.view(-1).repeat(gae.rollout.T) >= 0],
                       ref.rollout.rtg.view(-1)[ref.rollout.route.view(-1).repeat(ref.rollout.T) >= 0])
    bar = _grad_bar(mlp_mode)
    for a, b in ((ref.actor_net_cross, gae.actor_net_cross), (ref.actor_net_wait, gae.actor_net_wait),
                 (ref.critic_net_cross, gae.critic_net_cross), (ref.critic_net_wait, gae.critic_net_wait)):
        want, got = a.grad.double(), b.grad.double()
        scale = want.abs().max().item()
        assert scale > 0
        assert (got - want).abs().max().item() <= bar * scale, (got - want).abs().max().item() / scale
    for a, b in ((ref.actor_net_choice, gae.actor_net_choice), (ref.critic_net_choice, gae.critic_net_choice)):
        assert _bits_equal(a.grad, b.grad) and _bits_equal(a.flat, b.flat)


# ---------------------------------------------------------------------------------------------------------------------
# 3. a full GAE update against the float64 restatement

def _sd64(net):
    return {k: v.detach().double().cpu() for k, v in net.state_dict().items()}


def _gauss_lp(o, act, mean=-1.0, std=3.0, var=0.5):
    mu = torch.tanh(o) * std + mean
    return -(act - mu) ** 2 / (2 * var) - 0.5 * math.log(2 * math.pi * var)


def _reference_gae_update(algo, want, actor_sd, critic_sd, gamma, lam, epochs, dtype=torch.float64):
    """train_model_c in GAE mode in float64: V_old once from the critic before the update, R by the recursion, A = R - V_old
    normalised once; per epoch MSE(critic, R), clipped surrogate with the fixed A, torch.optim.Adam (PY:719-724).
    dtype = float32 gives what plain fp32 arithmetic achieves on the same buffers (the yardstick of DESIGN.md §4 for
    inputs with ±1e3 placeholder features, which the rollout's pair features contain)."""
    actor_sd, critic_sd = ({k: v.to(dtype) for k, v in sd.items()} for sd in (actor_sd, critic_sd))
    r = algo.rollout
    T, M = r.T, r.M
    cols = np.nonzero(r.route.view(-1).cpu().numpy() == want)[0]
    slots = (np.arange(T)[:, None] * M + cols[None, :]).reshape(-1)
    x = torch.as_tensor(r.obs_c.cpu().numpy()[:, slots].T, dtype=dtype)
    act = torch.as_tensor(r.act.cpu().numpy()[slots], dtype=dtype)
    logp_old = torch.as_tensor(r.logp.cpu().numpy()[slots], dtype=dtype)
    rew = r.rew.cpu().numpy().reshape(T, M)[:, cols]
    with torch.no_grad():
        V_old = _mlp64(critic_sd, x)[0][:, 0].numpy().reshape(T, len(cols))
    R = gae_returns(rew, V_old, gamma, lam).astype(V_old.dtype)
    A = torch.as_tensor((R - V_old).reshape(-1))
    An = (A - A.mean()) / (A.std() + 1e-10)
    Rt = torch.as_tensor(R.reshape(-1))
    pa = {k: v.clone().requires_grad_(True) for k, v in actor_sd.items()}
    pc = {k: v.clone().requires_grad_(True) for k, v in critic_sd.items()}
    oa, oc = torch.optim.Adam(list(pa.values()), lr=algo.actor_lr), torch.optim.Adam(list(pc.values()), lr=algo.critic_lr)
    out = dict(loss_a=[], loss_c=[], term_abs=[])
    for e in range(epochs):
        ratio = torch.exp(_gauss_lp(_mlp64(pa, x)[0][:, 0], act) - logp_old)
        terms = -torch.min(ratio * An, torch.clamp(ratio, 0.8, 1.2) * An)
        loss_a = terms.mean()
        loss_c = torch.mean((_mlp64(pc, x)[0][:, 0] - Rt) ** 2)
        oa.zero_grad(); oc.zero_grad()
        loss_a.backward(); loss_c.backward()
        if e == 0:
            out["grad_a"] = {k: v.grad.detach().clone() for k, v in pa.items()}
            out["grad_c"] = {k: v.grad.detach().clone() for k, v in pc.items()}
        oa.step(); oc.step()
        out["loss_a"].append(loss_a.item()); out["loss_c"].append(loss_c.item()); out["term_abs"].append(float(terms.detach().abs().mean()))
    out["actor"], out["critic"] = {k: v.detach() for k, v in pa.items()}, {k: v.detach() for k, v in pc.items()}
    return out


def test_gae_update_matches_fp64_restatement(mlp_mode):
    """lambda = 0.95, 10 epochs of the cross and wait pairs on a real rollout (scalable 4/3/2) against the float64
    restatement on the rollout's own buffers: losses every epoch, the first epoch's gradients, the weights after the update.
    The rollout's pair features include ±1e3 placeholders, so gradients, weights and the losses after the first epoch take
    the relaxed rule of DESIGN.md §4: the larger of the bar and 2x (FFMA) / 10x (auto) / 50x (tc) the deviation of the same
    update in plain fp32 (torch, CPU) from float64."""
    epochs, lam = 10, 0.95
    algo = _algo(1024, seed=11, gae_lambda=lam)
    pairs = ((0, algo.actor_net_cross, algo.critic_net_cross, algo.optimizer_actor_cross, algo.optimizer_critic_cross),
             (1, algo.actor_net_wait, algo.critic_net_wait, algo.optimizer_actor_wait, algo.optimizer_critic_wait))
    sd0 = {want: (_sd64(a), _sd64(c)) for want, a, c, _, _ in pairs}
    # Algo_PPO.update with the losses read after every epoch
    algo.rollout._set_head(algo.actor_net_cross)
    algo.rollout.futur_rewards()
    algo._prepare_gae()
    got = {want: dict(loss_a=[], loss_c=[]) for want, *_ in pairs}
    for e in range(epochs):
        for want, a, c, oa, oc in pairs:
            assert algo.train_model_c(a, c, oa, oc, want)
            loss = algo._loss.cpu().numpy()
            got[want]["loss_a"].append(loss[0]); got[want]["loss_c"].append(loss[1])
            if e == 0:
                got[want]["grad_a"], got[want]["grad_c"] = a.grad.double().cpu().numpy(), c.grad.double().cpu().numpy()
    assert _lib().mhppo_tc_failures() == 0
    bar = _grad_bar(mlp_mode)
    for want, a, c, _, _ in pairs:
        ref = _reference_gae_update(algo, want, *sd0[want], algo.gamma, lam, epochs)
        ref32 = _reference_gae_update(algo, want, *sd0[want], algo.gamma, lam, epochs, dtype=torch.float32)
        g = got[want]
        # 3xTF32 (mode auto) has 5x the FFMA bar for gradients (DESIGN.md §4); the fp32 yardstick scales with it.  In mode tc the
        # rollout's own inference also runs on the tensor cores, so the stored old log-probs carry its error on the ±1e3 rows
        # too (measured on a B200: wait actor 2.6e-3 of the largest gradient entry, fp32 autograd 1.2e-4): 25x.  From the second
        # epoch on, the losses also carry the divergence of the weights the earlier Adam steps took from those gradients.
        k32 = 2.0 * {0: 5.0, 1: 1.0, 2: 25.0}[mlp_mode]
        for e in range(epochs):
            la_lim = max(1e-5 * ref["term_abs"][e], k32 * abs(ref32["loss_a"][e] - ref["loss_a"][e]) if e else 0.0)
            lc_lim = max(1e-5 * ref["loss_c"][e], k32 * abs(ref32["loss_c"][e] - ref["loss_c"][e]) if e else 0.0)
            assert abs(g["loss_a"][e] - ref["loss_a"][e]) <= la_lim, ("actor loss", want, e, g["loss_a"][e], ref["loss_a"][e], la_lim)
            assert abs(g["loss_c"][e] - ref["loss_c"][e]) <= lc_lim, ("critic loss", want, e, g["loss_c"][e], ref["loss_c"][e], lc_lim)
        pk = lambda sd: _pack({k: v.double() for k, v in sd.items()}, 13).double().numpy()
        for k in ("grad_a", "grad_c"):
            w = pk(ref[k])
            err = np.abs(g[k] - w).max()
            lim = max(bar * np.abs(w).max(), k32 * np.abs(pk(ref32[k]) - w).max())
            assert err <= lim, (k, want, err / np.abs(w).max(), lim / np.abs(w).max())
        for net, key in ((a, "actor"), (c, "critic")):
            w = pk(ref[key])
            d = np.abs(net.flat.double().cpu().numpy() - w).max() / np.abs(w).max()
            # 1e-4 is the bar of DESIGN.md §4 for 4 epochs; the 3xTF32 path's error grows with the Adam steps, so 10 epochs of it
            # get 10/4 of that bar (measured on a B200: 1.02e-4 for the cross critic, 5e-5 for the actors)
            lim = max(1e-4 if mlp_mode == 1 else 2.5e-4, k32 * np.abs(pk(ref32[key]) - w).max() / np.abs(w).max())
            print("\nGAE update mode %d %s %s: weights %.3g of the largest (fp32 autograd %.3g)" % (
                mlp_mode, ("cross", "wait")[want], key, d, np.abs(pk(ref32[key]) - w).max() / np.abs(w).max()))
            assert d <= lim, ("weights", key, want, d, lim)


# ---------------------------------------------------------------------------------------------------------------------
# 4. mhppo_ppo_grad_ent against float64 autograd

ENT_WIDTHS = [12, 17, 18, 22, 30, 42, 54]


def _ent_qs():
    G, _ = _grid()
    return [127, 128, 129, 128 * G + 1, 256 * G - 1, 256 * G + 1, 384 * G + 5]


def _ent_case(L, ws, D, c, Q, seed, big_cols=False, saturate=None):
    rng = np.random.default_rng(seed)
    csd, asd = _net_sd(D, 1, 0, seed), _net_sd(D, 2, 2, seed + 1)
    if saturate:
        asd["layer4.weight"] = asd["layer4.weight"] * saturate
    b = _draw_batch(rng, Q, D, 2, csd, asd, big_cols=big_cols)
    CN = Q + 3
    cols = rng.permutation(CN)[:Q]
    x = np.full((D, CN), np.nan, np.float32); x[:, cols] = b["x"].T
    V32 = _mlp64({k: v.double() for k, v in csd.items()}, torch.as_tensor(b["x"], dtype=torch.float64))[0][:, 0].numpy().astype(np.float32)
    A = (b["rtg"] - V32).astype(np.float64)

    def buf(v):                                          # unselected slots NaN: a stray read poisons the result
        out = np.full(CN, np.nan, np.float32)
        out[cols] = v
        return torch.as_tensor(out, device="cuda")
    xd, rtg, Vd, act, logp = torch.as_tensor(x, device="cuda"), buf(b["rtg"]), buf(V32), buf(b["act"]), buf(b["logp"])
    idx = torch.as_tensor(cols.astype(np.int32), device="cuda")
    stats = torch.tensor([A.sum(), (A * A).sum(), float(Q)], dtype=torch.float64, device="cuda")
    net = _pack(asd, D).cuda()
    npar = L.mhppo_net_param_count(D)
    f0, f1 = float((b["act"] == 0).sum()) / Q, float((b["act"] == 1).sum()) / Q

    def launch(coef, dev_entry=False):
        g = torch.full((npar,), float("nan"), device="cuda")
        loss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
        args = (D, 2, xd.data_ptr(), D, CN, idx.data_ptr(), Q, CN, net.data_ptr(), act.data_ptr(), logp.data_ptr(), rtg.data_ptr(),
                Vd.data_ptr(), stats.data_ptr(), 1.0 / Q, f0, f1)
        if dev_entry:
            _check(L.mhppo_ppo_grad_dev(*args, g.data_ptr(), loss.data_ptr(), ws.data_ptr(), None))
        else:
            _check(L.mhppo_ppo_grad_ent(*args, coef, g.data_ptr(), loss.data_ptr(), ws.data_ptr(), None))
        torch.cuda.synchronize()
        return g.cpu(), loss.cpu()
    g1, l1 = launch(c)
    g2, l2 = launch(c)
    assert _bits_equal(g1, g2) and _bits_equal(l1, l2), "not repeatable"
    g0, l0 = launch(0.0)
    gd, ld = launch(0.0, dev_entry=True)
    assert _bits_equal(g0, gd) and _bits_equal(l0, ld), "ent_coef = 0 must be mhppo_ppo_grad_dev bit for bit"
    assert torch.isfinite(g1).all() and torch.isfinite(l1).all()
    loss, grads, term_abs = choice_loss_ent(asd, b["x"], A, b["act"], b["logp"], c)
    want = _pack(grads, D).double().numpy()
    got = g1.double().numpy()
    scale = np.abs(want).max()
    lim = 1e-5 * scale
    if big_cols:      # ±1e3 features: the larger of the bar and twice the error of plain fp32 autograd (DESIGN.md §4)
        _, g32, _ = choice_loss_ent(asd, b["x"], A, b["act"], b["logp"], c, dtype=torch.float32)
        lim = max(lim, 2 * np.abs(_pack(g32, D).double().numpy() - want).max())
    assert abs(l1.item() - loss) <= 1e-5 * term_abs, ("loss", D, c, Q, l1.item(), loss, term_abs)
    assert np.abs(got - want).max() <= lim, ("gradient", D, c, Q, np.abs(got - want).max() / max(scale, 1e-300))
    return got, want


@pytest.mark.parametrize("c", [0.01, 0.1])
@pytest.mark.parametrize("D", ENT_WIDTHS)
def test_ppo_grad_ent_matches_fp64(lib0, ws, D, c):
    """Every choice width (KP 16 / 32 / 56) at the tile and grid boundaries of k_ppo_grad<KP, 2>: 1 or 2 samples per thread,
    CTAs with 0, 1, 2 and 3+ tiles."""
    for i, Q in enumerate(_ent_qs()):
        _ent_case(lib0, ws, D, c, Q, seed=100 * D + 10 * i + int(c * 100))


@pytest.mark.parametrize("D", [18, 30])
def test_ppo_grad_ent_placeholder_features(lib0, ws, D):
    G, _ = _grid()
    _ent_case(lib0, ws, D, 0.1, 128 * G + 77, seed=7 + D, big_cols=True)


def test_ppo_grad_ent_saturated_logits(lib0, ws):
    """Logits hundreds to thousands apart (p = 0 exactly for many samples): a finite loss and gradient that match."""
    G, _ = _grid()
    got, want = _ent_case(lib0, ws, 30, 0.1, 128 * G + 5, seed=5, saturate=300.0)
    assert np.isfinite(got).all()


def test_ppo_grad_ent_rejects_invalid_arguments(lib0, ws):
    L = lib0
    D, Q = 30, 40
    x = torch.zeros(D * Q, device="cuda")
    v = torch.zeros(Q, device="cuda")
    st = torch.tensor([0.0, 1.0, float(Q)], dtype=torch.float64, device="cuda")
    g = torch.zeros(L.mhppo_net_param_count(D), device="cuda")
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    net = torch.zeros(L.mhppo_net_param_count(D), device="cuda")

    def call(head, coef, n_in=D):
        return L.mhppo_ppo_grad_ent(n_in, head, x.data_ptr(), min(D, n_in), Q, None, Q, Q, net.data_ptr(), v.data_ptr(), v.data_ptr(),
                                    v.data_ptr(), v.data_ptr(), st.data_ptr(), 1.0 / Q, 0.5, 0.5, coef, g.data_ptr(), loss.data_ptr(),
                                    ws.data_ptr(), None)
    for coef in (math.nan, math.inf, -math.inf):
        assert call(2, coef) == EINVAL
    for head in (0, 1):
        assert call(head, 0.01, n_in=13) == EINVAL
        assert call(head, 0.0, n_in=13) == 0
    assert call(2, 0.01) == 0 and call(2, -0.01) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 5. smoke run, options validation

def test_train_with_options_stays_finite(mlp_mode):
    algo = _algo(26, seed=2, nb=(1, 1, 1), gae_lambda=0.95, entropy_coef=0.01)
    algo.train(20, save_traces=False)
    torch.cuda.synchronize()
    for _, _, net in algo._nets():
        assert torch.isfinite(net.flat).all()
    assert _lib().mhppo_tc_failures() == 0


def test_algo_rejects_bad_options(lib0):
    import mhppo_b200 as mh
    env = mh.VecCrosswalkEnv("coop_scalable", 8, nb_car=1, nb_ped=1, nb_lines=1, seed=1, env_id0=0)
    kw = dict(num_states_c=13, num_states_d=18, num_actions=1, mean=-1.0, std=3.0, nb_cars=1, dt=0.3)
    for bad in (dict(gae_lambda=-0.1), dict(gae_lambda=1.01), dict(gae_lambda=math.nan), dict(gae_lambda="0.9"), dict(gae_lambda=True),
                dict(gae_lambda=0.9, gamma=1.5), dict(entropy_coef=math.inf), dict(entropy_coef=math.nan), dict(entropy_coef=-0.01),
                dict(entropy_coef=None)):
        with pytest.raises(ValueError):
            mh.Algo_PPO(mh.Model_PPO, env, **kw, **bad)
    a = mh.Algo_PPO(mh.Model_PPO, env, **kw, gae_lambda=0, entropy_coef=0)
    assert a.rollout.ret is None                       # GAE buffers are allocated by the first GAE update only


# ---------------------------------------------------------------------------------------------------------------------
# 6. two ranks == one rank, with both options on

def test_two_rank_gae_entropy_equals_one_rank(lib0):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29519", os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "OK" in r.stdout


def _dist_main():
    """R ranks of N/R envs with disjoint env ids against one rank of N envs, GAE (lambda 0.95) + entropy bonus (0.01):
    bit-identical rollout buffers and GAE returns on the shard, weights within 1e-4 (tests/dist_ppo_check.py)."""
    import torch.distributed as dist
    import mhppo_b200
    from mhppo_b200 import ppo
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    N = 4096
    n = N // world

    def run(N, env_id0, use_dist):
        ppo.set_distributed(use_dist)
        env = mhppo_b200.VecCrosswalkEnv("coop_scalable", N, nb_car=4, nb_ped=3, nb_lines=2, seed=77, env_id0=env_id0, device=dev)
        torch.manual_seed(0 if not use_dist else 1000 * rank)
        algo = mhppo_b200.Algo_PPO(mhppo_b200.Model_PPO, env, num_states_c=13, num_states_d=30, num_actions=1, mean=-1.0, std=3.0,
                                   nb_cars=4, dt=0.3, gae_lambda=0.95, entropy_coef=0.01)
        algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        algo.update(epochs=3)
        torch.cuda.synchronize()
        return algo
    sharded = run(n, rank * n, True)
    whole = run(N, 0, False)
    r_s, r_w = sharded.rollout, whole.rollout
    T, C = r_s.T, r_s.C
    for name in ("act", "logp", "rew", "rtg", "ret"):
        a = getattr(r_s, name).view(T, C, n)
        b = getattr(r_w, name).view(T, C, N)[:, :, rank * n:(rank + 1) * n]
        assert torch.equal(a, b), "rollout buffer %s differs on rank %d" % (name, rank)
    worst = 0.0
    for (_, _, ns), (_, _, nw) in zip(sharded._nets(), whole._nets()):
        worst = max(worst, (ns.flat - nw.flat).abs().max().item() / max(nw.flat.abs().max().item(), 1e-12))
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("two-rank GAE + entropy world=%d: rollout shards bit-identical, max relative weight difference %.3e" % (world, t.item()))
    assert t.item() < 1e-4, t.item()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    _dist_main()
