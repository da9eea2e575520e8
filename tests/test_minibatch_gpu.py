"""The minibatch option of the update on the GPU: mhppo_minibatch_plan through the C ABI and Algo_PPO(n_minibatches=B) on real
rollouts, against the numpy restatement of tests/test_minibatch.py and a float64 restatement of the minibatch update.

Bars (DESIGN.md §4): the plan exactly; B = 1 bit for bit against the default path; a 3-epoch x 3-minibatch update (9 steps per
net, within the 10-step bars) with the bars and the relaxed ±1e3 rule of tests/test_gae_entropy_gpu.py.  The PPO-level cases run
in the three mhppo_set_mlp_mode modes.  Run as a script under torch.distributed.run it is the two-rank check of the option."""
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

from test_gae_entropy import gae_returns  # noqa: E402
from test_minibatch import minibatch_plan  # noqa: E402
from test_update_kernels_gpu import _mlp64, _pack, _bits_equal  # noqa: E402

pytestmark = pytest.mark.gpu
EINVAL = -1
CAP = 1024


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


# ---------------------------------------------------------------------------------------------------------------------
# 1. mhppo_minibatch_plan against the restatement, exactly

def _plan_gpu(L, route, exist, act_d, seed, env_id0, iteration, E, B):
    from mhppo_b200._lib import RolloutCfg
    import ctypes as C
    Cn, N = route.shape
    cfg = RolloutCfg(nb_ped=1, nb_lines=1, T=80, legacy_nb_car=Cn, n_envs=N, seed=seed, env_id0=env_id0)
    M = Cn * N
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    rd, ed, ad = d(route), d(exist), d(act_d.astype(np.float32))
    lists = torch.full((E, 3, M), -7, dtype=torch.int32, device="cuda")
    off = torch.full((E, 3, B + 1), -7, dtype=torch.int64, device="cuda")
    cnt = torch.full((E, 5, B), -7, dtype=torch.int64, device="cuda")
    ws = torch.empty(1280 * E * B, dtype=torch.uint8, device="cuda")
    _check(L.mhppo_minibatch_plan(C.byref(cfg), rd.data_ptr(), ed.data_ptr(), ad.data_ptr(), iteration, E, B, lists.data_ptr(),
                                  off.data_ptr(), cnt.data_ptr(), ws.data_ptr(), None))
    torch.cuda.synchronize()
    return lists.cpu().numpy(), off.cpu().numpy(), cnt.cpu().numpy()


def _inputs(Cn, N, seed, absent=False):
    rng = np.random.default_rng(seed)
    route = rng.choice(np.array([-1, 0, 1], np.int8), (Cn, N), p=[0.25, 0.45, 0.3])
    if absent:
        route[:] = -1
    exist = (route >= 0).astype(np.int8)
    act_d = rng.integers(0, 2, (Cn, N)).astype(np.float32)
    return route, exist, act_d


def _check_plan(got, want, E):
    lists, off, cnt = got
    L, woff, wcnt = want
    assert np.array_equal(off, woff) and np.array_equal(cnt, wcnt)
    for e in range(E):
        for s in range(3):
            assert np.array_equal(lists[e, s, :woff[e, s, -1]], L[e][s]), (e, s)


@pytest.mark.parametrize("E", [1, 10])
@pytest.mark.parametrize("B", [1, 2, 7, CAP])
@pytest.mark.parametrize("N", [1, 26, 255, 256, 257, 131072])
@pytest.mark.parametrize("Cn", [1, 4])
def test_plan_matches_restatement(lib0, Cn, N, B, E):
    for k, (seed, env_id0, it) in enumerate(((3, 0, 0), (2 ** 35 + 9, 1000003, 41), (77, 2 ** 33 - 5, 299))):
        if N == 131072 and k:
            break
        route, exist, act_d = _inputs(Cn, N, seed=N + B + k)
        got = _plan_gpu(lib0, route, exist, act_d, seed, env_id0, it, E, B)
        _check_plan(got, minibatch_plan(route, exist, act_d, seed, env_id0, it, E, B), E)
        again = _plan_gpu(lib0, route, exist, act_d, seed, env_id0, it, E, B)
        assert all(np.array_equal(a, b) for a, b in zip(got, again)), "not repeatable"


@pytest.mark.parametrize("B", [1, 64, CAP])
def test_plan_all_absent_and_more_buckets_than_columns(lib0, B):
    for Cn, N, absent in ((4, 300, True), (1, 26, False), (4, 7, False)):
        route, exist, act_d = _inputs(Cn, N, seed=B + N, absent=absent)
        got = _plan_gpu(lib0, route, exist, act_d, 5, 11, 2, 3, B)
        _check_plan(got, minibatch_plan(route, exist, act_d, 5, 11, 2, 3, B), 3)
        if absent:
            assert not got[2].any() and not got[1].any()


@pytest.mark.parametrize("B", [4, 7])
def test_plan_sharded_equals_whole(lib0, B):
    """The plan of envs [r*n, (r+1)*n) called with env_id0 = r*n is the matching part of the plan of all envs, bucket by bucket."""
    Cn, N, R, E, seed, it = 4, 4096, 4, 3, 77, 5
    n = N // R
    route, exist, act_d = _inputs(Cn, N, seed=1)
    lists, off, cnt = _plan_gpu(lib0, route, exist, act_d, seed, 0, it, E, B)
    total = np.zeros_like(cnt)
    for r in range(R):
        sl = slice(r * n, (r + 1) * n)
        ls, os_, cs = _plan_gpu(lib0, route[:, sl], exist[:, sl], act_d[:, sl], seed, r * n, it, E, B)
        total += cs
        for e in range(E):
            for s in range(3):
                for b in range(B):
                    whole = lists[e, s, off[e, s, b]:off[e, s, b + 1]]
                    env = whole % N
                    part = whole[(env >= r * n) & (env < (r + 1) * n)]
                    mine = ls[e, s, os_[e, s, b]:os_[e, s, b + 1]]
                    assert np.array_equal((mine // n) * N + mine % n + r * n, part), (r, e, s, b)
    assert np.array_equal(total, cnt)


def test_plan_rejects_invalid_arguments(lib0):
    from mhppo_b200._lib import RolloutCfg
    import ctypes as C
    L = lib0
    cfg = RolloutCfg(nb_ped=1, nb_lines=1, T=80, legacy_nb_car=2, n_envs=10, seed=1, env_id0=0)
    i8 = torch.zeros(20, dtype=torch.int8, device="cuda")
    f = torch.zeros(20, device="cuda")
    big = torch.zeros(1 << 22, dtype=torch.int64, device="cuda")
    p = dict(route=i8.data_ptr(), exist=i8.data_ptr(), act=f.data_ptr(), lists=big.data_ptr(), off=big.data_ptr(), cnt=big.data_ptr(),
             ws=big.data_ptr())

    def call(E=2, B=4, cfgp=True, **null):
        q = {k: (None if null.get(k) else v) for k, v in p.items()}
        return L.mhppo_minibatch_plan(C.byref(cfg) if cfgp else None, q["route"], q["exist"], q["act"], 0, E, B, q["lists"], q["off"],
                                      q["cnt"], q["ws"], None)
    for k in p:
        assert call(**{k: True}) == EINVAL, k
    assert call(cfgp=False) == EINVAL
    for bad in (dict(E=0), dict(E=-1), dict(B=0), dict(B=-3), dict(B=CAP + 1)):
        assert call(**bad) == EINVAL, bad
    assert call(B=1) == 0 and call(B=CAP, E=1) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 2. B = 1 is the default path, bit for bit

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


@pytest.mark.parametrize("opts", [{}, dict(gae_lambda=0.95), dict(entropy_coef=0.01)], ids=["reference", "gae", "entropy"])
def test_one_minibatch_is_default_path_bitwise(mlp_mode, opts):
    ref, mb = _algo(2048, **opts), _algo(2048, n_minibatches=1, **opts)
    ref.update(epochs=3)
    mb.update(epochs=3)
    torch.cuda.synchronize()
    for (_, _, a), (_, _, b) in zip(ref._nets(), mb._nets()):
        assert a.step == b.step == 3
        for t in ("flat", "m", "v"):
            assert _bits_equal(getattr(a, t), getattr(b, t)), t


# ---------------------------------------------------------------------------------------------------------------------
# 3. a minibatch update against the float64 restatement

def _sd64(net):
    return {k: v.detach().double().cpu() for k, v in net.state_dict().items()}


def _gauss_lp(o, act, mean=-1.0, std=3.0, var=0.5):
    mu = torch.tanh(o) * std + mean
    return -(act - mu) ** 2 / (2 * var) - 0.5 * math.log(2 * math.pi * var)


def _normalise(A):
    return (A - A.mean()) / (A.std() + 1e-10)


def _reference_mb_update(algo, which, actor_sd, critic_sd, epochs, B, lam=None, c=0.0, dtype=torch.float64):
    """The minibatch update of one pair (which = 0 cross, 1 wait, 2 choice) in `dtype` on the rollout's own buffers, with the
    minibatches of the numpy plan restatement: per minibatch with >= 2 samples, reference mode takes V from the current critic
    and normalises A = rtg - V over the minibatch; GAE mode uses the whole update's returns and normalised advantages; the choice
    pair uses the minibatch's action fractions and, if c > 0, the entropy bonus; one Adam step per pair and minibatch."""
    r = algo.rollout
    T, M = r.T, r.M
    route, exist, act_d = r.route.cpu().numpy(), r.exist.cpu().numpy(), r.act_d.cpu().numpy().reshape(r.C, r.N)
    plan, off, _ = minibatch_plan(route, exist, act_d, algo.env._seed, algo.env._env_id0, r.iteration - 1, epochs, B)
    pa = {k: v.to(dtype).clone().requires_grad_(True) for k, v in actor_sd.items()}
    pc = {k: v.to(dtype).clone().requires_grad_(True) for k, v in critic_sd.items()}
    oa = torch.optim.Adam(list(pa.values()), lr=algo.actor_d_lr if which == 2 else algo.actor_lr)
    oc = torch.optim.Adam(list(pc.values()), lr=algo.critic_d_lr if which == 2 else algo.critic_lr)
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=dtype)
    if which == 2:
        obs, ret, act, logp = r.obs_d.cpu().numpy(), r.rew_d.cpu().numpy(), r.act_d.cpu().numpy(), r.logp_d.cpu().numpy()
    else:
        obs, ret, act, logp = r.obs_c.cpu().numpy(), r.rtg.cpu().numpy(), r.act.cpu().numpy(), r.logp.cpu().numpy()
    if lam is not None:                   # GAE: V_old once, the returns and the advantages normalised over the whole update
        cols = np.nonzero(route.reshape(-1) == which)[0]
        slots = (np.arange(T)[:, None] * M + cols[None, :]).reshape(-1)
        with torch.no_grad():
            V_old = _mlp64(pc, t(obs[:, slots].T))[0][:, 0].numpy().reshape(T, len(cols))
        R = gae_returns(r.rew.cpu().numpy().reshape(T, M)[:, cols], V_old, algo.gamma, lam)
        ret = np.zeros(T * M); ret[slots] = R.reshape(-1)
        An_all = np.zeros(T * M); An_all[slots] = _normalise(t((R - V_old).reshape(-1))).numpy()
    out = dict(loss_a=[], loss_c=[], term_abs=[])
    for e in range(epochs):
        for b in range(B):
            cols = plan[e][which][off[e, which, b]:off[e, which, b + 1]]
            slots = cols if which == 2 else (np.arange(T)[:, None] * M + cols[None, :]).reshape(-1)
            n = len(slots)
            if n < 2:
                continue
            x = t(obs[:, slots].T)
            if lam is not None:
                An = t(An_all[slots])
            else:
                with torch.no_grad():
                    An = _normalise(t(ret[slots]) - _mlp64(pc, x)[0][:, 0])
            o = _mlp64(pa, x)[0]
            if which == 2:
                lp = torch.log_softmax(o[:, :2], dim=1)
                ratio = torch.exp(lp - t(logp[slots])[:, None])
                surr = -torch.min(ratio * An[:, None], torch.clamp(ratio, 0.8, 1.2) * An[:, None])
                a = act[slots]
                f = t([float((a == k).sum()) / n for k in (0, 1)])
                terms = (surr * f).sum(1) + c * (torch.exp(lp) * lp).sum(1)
            else:
                ratio = torch.exp(_gauss_lp(o[:, 0], t(act[slots])) - t(logp[slots]))
                terms = -torch.min(ratio * An, torch.clamp(ratio, 0.8, 1.2) * An)
            loss_a = terms.mean()
            loss_c = torch.mean((_mlp64(pc, x)[0][:, 0] - t(ret[slots])) ** 2)
            oa.zero_grad(); oc.zero_grad()
            loss_a.backward(); loss_c.backward()
            if "grad_a" not in out:
                out["grad_a"] = {k: v.grad.detach().clone() for k, v in pa.items()}
                out["grad_c"] = {k: v.grad.detach().clone() for k, v in pc.items()}
            oa.step(); oc.step()
            out["loss_a"].append(loss_a.item()); out["loss_c"].append(loss_c.item()); out["term_abs"].append(float(terms.detach().abs().mean()))
    out["actor"], out["critic"] = {k: v.detach() for k, v in pa.items()}, {k: v.detach() for k, v in pc.items()}
    return out


def _record(algo):
    """Wrap the epoch bodies so that every minibatch's losses (and the first minibatch's gradients) of each pair are kept."""
    got = {w: dict(loss_a=[], loss_c=[]) for w in (0, 1, 2)}
    ec, ed = algo._epoch_c, algo._epoch_d

    def keep(w, actor, critic):
        g = got[w]
        loss = algo._loss.cpu().numpy()
        g["loss_a"].append(loss[0]); g["loss_c"].append(loss[1])
        if "grad_a" not in g:
            g["grad_a"], g["grad_c"] = actor.grad.double().cpu().numpy(), critic.grad.double().cpu().numpy()

    def c_(actor, critic, oa, oc, want, *a):
        ec(actor, critic, oa, oc, want, *a); keep(want, actor, critic)

    def d_(actor, critic, oa, oc, *a):
        ed(actor, critic, oa, oc, *a); keep(2, actor, critic)
    algo._epoch_c, algo._epoch_d = c_, d_
    return got


@pytest.mark.parametrize("case", ["reference", "gae", "choice", "choice_entropy"])
def test_minibatch_update_matches_fp64_restatement(mlp_mode, case):
    """3 epochs x 3 minibatches on a real rollout (scalable 4/3/2) against the float64 restatement: losses of every minibatch,
    the first minibatch's gradients, the weights after the update.  The relaxed rule of tests/test_gae_entropy_gpu.py applies
    (the larger of the bar and k x the deviation of the same update in plain fp32); mode tc's cross / wait actors take the wider
    bars below.  Every deviation is printed before the check."""
    epochs, B = 3, 3
    lam = 0.95 if case == "gae" else None
    c = 0.01 if case == "choice_entropy" else 0.0
    algo = _algo(1024, seed=11, n_minibatches=B, gae_lambda=lam, entropy_coef=c)
    pairs = {0: (algo.actor_net_cross, algo.critic_net_cross), 1: (algo.actor_net_wait, algo.critic_net_wait),
             2: (algo.actor_net_choice, algo.critic_net_choice)}
    whiches = (2,) if case.startswith("choice") else (0, 1)
    sd0 = {w: (_sd64(a), _sd64(cn)) for w, (a, cn) in pairs.items()}
    got = _record(algo)
    algo.update(epochs=epochs)
    torch.cuda.synchronize()
    assert _lib().mhppo_tc_failures() == 0
    uses_tc = mlp_mode in (0, 2)
    k32 = 2.0 * ({0: 5.0, 1: 1.0, 2: 25.0}[mlp_mode] if not whiches == (2,) else 1.0)
    bar = 5e-5 if (uses_tc and whiches != (2,)) else 1e-5
    fails = []
    for w in whiches:
        a, cn = pairs[w]
        ref = _reference_mb_update(algo, w, *sd0[w], epochs, B, lam=lam, c=c)
        ref32 = _reference_mb_update(algo, w, *sd0[w], epochs, B, lam=lam, c=c, dtype=torch.float32)
        g = got[w]
        assert len(g["loss_a"]) == len(ref["loss_a"]) == a.step == cn.step > 0
        for i in range(len(ref["loss_a"])):
            # after the first step the losses also carry the weights' divergence from the earlier steps: in the tensor-core modes
            # the 3xTF32 gradient bar (5x the FFMA bar) applies to them
            lb = 1e-5 if i == 0 else bar
            for k, scale in (("loss_a", ref["term_abs"][i]), ("loss_c", ref["loss_c"][i])):
                dev = abs(g[k][i] - ref[k][i])
                lim = max(lb * scale, k32 * abs(ref32[k][i] - ref[k][i]) if i else 0.0)
                print("mode %d %s pair %d %s minibatch %d: %.3g of the scale (limit %.3g)" % (mlp_mode, case, w, k, i, dev / scale, lim / scale))
                if dev > lim:
                    fails.append((k, w, i, dev / scale, lim / scale))
        D = 13 if w < 2 else algo.rollout.shape_env_d
        pk = lambda sd: _pack({k: v.double() for k, v in sd.items()}, D).double().numpy()
        for k in ("grad_a", "grad_c"):
            want = pk(ref[k])
            scale = np.abs(want).max()
            err, err32 = np.abs(g[k] - want).max() / scale, np.abs(pk(ref32[k]) - want).max() / scale
            lim = max(bar, k32 * err32)
            if mlp_mode == 2 and w < 2 and k == "grad_a":
                # mode tc runs the rollout inference on the tensor cores too: its error on the ±1e3 placeholder rows sits in the
                # stored old log-probs (DESIGN.md §4), and a minibatch of 1/B of the samples gives those rows B times the weight of
                # the full batch (full batch: 2.6e-3 of the largest wait-actor entry; measured here on a B200: 5.7e-3 and 7.0e-3)
                lim = max(lim, 1e-2)
            print("mode %d %s pair %d %s: %.3g of the largest entry (fp32 autograd %.3g, limit %.3g)" % (mlp_mode, case, w, k, err, err32, lim))
            if err > lim:
                fails.append((k, w, err, lim))
        for net, key in ((a, "actor"), (cn, "critic")):
            want = pk(ref[key])
            d = np.abs(net.flat.double().cpu().numpy() - want).max() / np.abs(want).max()
            d32 = np.abs(pk(ref32[key]) - want).max() / np.abs(want).max()
            lim = max(2.5e-4 if uses_tc and w < 2 else 1e-4, k32 * d32)
            if mlp_mode == 2 and w < 2 and key == "actor":
                lim = max(lim, 2e-3)         # the same rows after 9 steps (measured on a B200: 9.7e-4 and 1.06e-3 for the wait actor)
            print("mode %d %s pair %d %s weights: %.3g of the largest (fp32 autograd %.3g, limit %.3g)" % (mlp_mode, case, w, key, d, d32, lim))
            if d > lim:
                fails.append(("weights", key, w, d, lim))
    assert not fails, fails


# ---------------------------------------------------------------------------------------------------------------------
# 4. determinism, 5. the skip rule, 6. options

def test_minibatch_update_is_deterministic(mlp_mode):
    a, b = _algo(2048, n_minibatches=4, gae_lambda=0.95, entropy_coef=0.01), _algo(2048, n_minibatches=4, gae_lambda=0.95, entropy_coef=0.01)
    a.update(epochs=3)
    b.update(epochs=3)
    torch.cuda.synchronize()
    for (_, _, x), (_, _, y) in zip(a._nets(), b._nets()):
        assert x.step == y.step and _bits_equal(x.flat, y.flat) and _bits_equal(x.m, y.m) and _bits_equal(x.v, y.v)


def test_skip_rule_step_counts(mlp_mode):
    """26 envs at 1/1/1 with B = 64 (most buckets empty): each net takes one Adam step per (epoch, minibatch) with >= 2 samples."""
    E, B = 10, 64
    algo = _algo(26, seed=2, nb=(1, 1, 1), n_minibatches=B)
    r = algo.rollout
    _, _, cnt = minibatch_plan(r.route.cpu().numpy(), r.exist.cpu().numpy(), r.act_d.cpu().numpy().reshape(r.C, r.N), algo.env._seed,
                               algo.env._env_id0, r.iteration - 1, E, B)
    algo.update(epochs=E)
    torch.cuda.synchronize()
    want = [int((r.T * cnt[:, 0] >= 2).sum()), int((r.T * cnt[:, 1] >= 2).sum()), int((cnt[:, 2] >= 2).sum())]
    assert sum(want) > 0
    for w, (a, c) in enumerate(((algo.actor_net_cross, algo.critic_net_cross), (algo.actor_net_wait, algo.critic_net_wait),
                                (algo.actor_net_choice, algo.critic_net_choice))):
        assert a.step == c.step == want[w], (w, a.step, want[w])
    algo.train(20, save_traces=False)
    torch.cuda.synchronize()
    for _, _, net in algo._nets():
        assert torch.isfinite(net.flat).all()


def test_algo_rejects_bad_minibatch_options(lib0):
    import mhppo_b200 as mh
    env = mh.VecCrosswalkEnv("coop_scalable", 8, nb_car=1, nb_ped=1, nb_lines=1, seed=1, env_id0=0)
    kw = dict(num_states_c=13, num_states_d=18, num_actions=1, mean=-1.0, std=3.0, nb_cars=1, dt=0.3)
    for bad in (True, False, 2.0, 0.5, 0, -1, -64, CAP + 1, 10 ** 9, "4", math.nan):
        with pytest.raises(ValueError):
            mh.Algo_PPO(mh.Model_PPO, env, **kw, n_minibatches=bad)
    for good in (None, 1, 7, CAP, np.int64(16)):
        assert mh.Algo_PPO(mh.Model_PPO, env, **kw, n_minibatches=good).n_minibatches == good


# ---------------------------------------------------------------------------------------------------------------------
# 7. two ranks == one rank, B = 4

def test_two_rank_minibatches_equal_one_rank(lib0):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29523", os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "OK" in r.stdout


def _dist_main():
    """R ranks of N/R envs with disjoint env ids against one rank of N envs, B = 4 minibatches, reference mode: the same step
    counts and weights within 1e-4."""
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
                                   nb_cars=4, dt=0.3, n_minibatches=4)
        algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        algo.update(epochs=3)
        torch.cuda.synchronize()
        return algo
    sharded = run(n, rank * n, True)
    whole = run(N, 0, False)
    worst = 0.0
    for (_, _, ns), (_, _, nw) in zip(sharded._nets(), whole._nets()):
        assert ns.step == nw.step, (ns.step, nw.step)
        worst = max(worst, (ns.flat - nw.flat).abs().max().item() / max(nw.flat.abs().max().item(), 1e-12))
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("two-rank minibatches world=%d: same step counts, max relative weight difference %.3e" % (world, t.item()))
    assert t.item() < 1e-4, t.item()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    _dist_main()
