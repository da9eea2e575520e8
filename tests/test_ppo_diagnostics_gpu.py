"""The update diagnostics on the GPU (Algo_PPO(diagnostics=True, target_kl=delta), mhppo_critic_grad_diag / mhppo_ppo_grad_diag /
mhppo_adam2_halt): bit-identical updates with and without them, the record of every step against a float64 restatement at the
parameters before that step, the kernels alone at every input width, tile / grid boundary and on ±1e3 placeholder rows, the
target-KL halt against a non-halting run, determinism, and (two GPUs) two ranks against one.

Bars (DESIGN.md §4 "Diagnostics"): approx_kl, entropy and the explained variance within 1e-5 relative; only a batch that has
±1e3 placeholder rows takes the relaxed rule, the larger of that and k x the deviation of the same restatement in plain fp32
(k of tests/test_minibatch_gpu.py: 2 x 1 / 5 / 25 for modes ffma / auto / tc); only the first step of a pair takes, for approx_kl,
the absolute floor `_k3_floor` (a few fp32 roundings of log r, which is what the first step's KL is made of).  The clip count
exactly, except for samples whose float64 ratio lies within 1e-5 of 0.8 or 1.2 (on a ±1e3 row: within the larger of 1e-5 and k x
the fp32 restatement's ratio error): the counts may differ by at most their number."""
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

from test_ppo_diagnostics import k3  # noqa: E402
from test_update_kernels_gpu import _mlp64, _pack, _bits_equal, _net_sd, _draw_batch, _layout, _scatter, _grid, DEFAULT_HEAD  # noqa: E402

pytestmark = pytest.mark.gpu
EPS32 = 2.0 ** -24
K32 = {0: 10.0, 1: 2.0, 2: 50.0}


def _lib():
    import mhppo_b200
    return mhppo_b200.lib()


def _check(rc):
    from mhppo_b200._lib import check
    check(rc)


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


def _state(algo):
    return [(n.step, n.flat.clone(), n.m.clone(), n.v.clone()) for _, _, n in algo._nets()]


def _same_state(a, b):
    return all(x[0] == y[0] and all(_bits_equal(p, q) for p, q in zip(x[1:], y[1:])) for x, y in zip(a, b))


# ---------------------------------------------------------------------------------------------------------------------
# 1. diagnostics change no bit of the update

SETTINGS = {"full": {}, "B4": dict(n_minibatches=4), "gae_entropy": dict(gae_lambda=0.95, entropy_coef=0.01)}


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_diagnostics_leave_the_update_bit_identical(mlp_mode, setting):
    opts = SETTINGS[setting]
    ref = _algo(2048, **opts)
    ref.update()
    loss_ref = ref._loss.clone()
    torch.cuda.synchronize()
    for extra in (dict(diagnostics=True), dict(target_kl=1e9)):
        a = _algo(2048, **opts, **extra)
        a.update()
        torch.cuda.synchronize()
        assert _same_state(_state(ref), _state(a)), extra
        assert _bits_equal(loss_ref, a._loss), extra
        st = a.last_update_stats
        assert set(st) == {"cross", "wait", "choice"}
        for p, arr in st.items():
            assert len(arr) > 0 and arr["taken"].all(), (p, extra)
            assert np.isfinite(arr["approx_kl"]).all() and (arr["approx_kl"] >= 0).all()
            assert np.isnan(arr["entropy"]).all() == (p != "choice")


# ---------------------------------------------------------------------------------------------------------------------
# 2. the record of every step against the float64 restatement

def _sd(net, dtype=torch.float64):
    return {k: v.detach().to(dtype).cpu() for k, v in net.state_dict().items()}


def _capture(algo):
    """Wrap the epoch bodies: per pair, the parameters before each step and the step's columns."""
    steps = {0: [], 1: [], 2: []}
    ec, ed = algo._epoch_c, algo._epoch_d

    def cols_of(idx, K):
        cands = [v[0] for k, v in algo._sel_cache.items() if k in (0, 1, None)] + ([algo._mb["lists"]] if "lists" in algo._mb else [])
        for t in cands:
            base = t.data_ptr()
            if base <= idx < base + 4 * t.numel():
                o = (idx - base) // 4
                return t[o:o + K].cpu().numpy().astype(np.int64)
        raise AssertionError("unknown column list")

    def c_(actor, critic, oa, oc, want, idx, K, n):
        steps[want].append(dict(a=_sd(actor), c=_sd(critic), cols=cols_of(idx, K), n=n))
        ec(actor, critic, oa, oc, want, idx, K, n)

    def d_(actor, critic, oa, oc, idx, K, n, fr):
        steps[2].append(dict(a=_sd(actor), c=_sd(critic), cols=cols_of(idx, K), n=n))
        ed(actor, critic, oa, oc, idx, K, n, fr)
    algo._epoch_c, algo._epoch_d = c_, d_
    return steps


def _restate(x, R, act, logp_old, asd, csd, head, dtype):
    """Per-sample log r, fp64 ratio, entropy (head 2), V of one step in `dtype` (inputs: fp32 numpy arrays, x [n, D])."""
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=dtype)
    with torch.no_grad():
        xx = t(x)
        V = _mlp64({k: v.to(dtype) for k, v in csd.items()}, xx)[0][:, 0]
        o = _mlp64({k: v.to(dtype) for k, v in asd.items()}, xx)[0]
        if head == 2:
            lsm = torch.log_softmax(o[:, :2], dim=1)
            lpa = lsm.gather(1, t(act).long()[:, None])[:, 0]
            H = -(torch.exp(lsm) * lsm).sum(1)
        else:
            mean, std, var = DEFAULT_HEAD
            mu = torch.tanh(o[:, 0]) * std + mean
            lpa = -(t(act) - mu) ** 2 / (2 * var) - 0.5 * math.log(2 * math.pi * var)
            H = None
        log_r = lpa - t(logp_old)
    f = lambda v: None if v is None else v.double().numpy()
    return dict(log_r=f(log_r), lp=f(lpa), V=f(V), H=f(H), R=np.asarray(R, np.float64))


def _k3_floor(ref, ref32, logp_old, k):
    """Absolute bar of the mean k3: the kernel's fp32 log r carries an error u_s of a few fp32 roundings of its two terms (or
    k x the fp32 restatement's own error), and |k3(l + u) - k3(l)| <= |expm1(l)| u + e^(|l| + u) u^2 / 2."""
    l = ref["log_r"]
    u = np.maximum(8 * EPS32 * (np.abs(ref["lp"]) + np.abs(np.asarray(logp_old, np.float64))), k * np.abs(ref32["log_r"] - l))
    return float(np.mean(np.abs(np.expm1(l)) * u + np.exp(np.minimum(np.abs(l) + u, 700)) * u * u / 2))


def _ev(R, V):
    vr = R.var()
    return 1.0 - (R - V).var() / vr if vr > 0 else float("nan")


def _compare(got, x, R, act, logp_old, asd, csd, head, k, tag, fails, first=False):
    """got: (approx_kl, clip count, entropy, explained variance) of the kernel; the rest restated here.  The bars are 1e-5 relative
    and the exact clip count with the 1e-5 window.  Only a batch with ±1e3 feature rows takes the relaxed rule (k x the deviation
    of the fp32 restatement; for the clip window, per ±1e3 row), and only the first step of a pair (`first`) the absolute
    approx_kl floor of _k3_floor."""
    ref, ref32 = (_restate(x, R, act, logp_old, asd, csd, head, d) for d in (torch.float64, torch.float32))
    n = len(R)
    big = np.abs(np.asarray(x)).max(axis=1) >= 999.0 if len(R) else np.zeros(0, bool)     # the ±1e3 placeholder rows
    kr = k if big.any() else 0.0
    kl, kl32 = k3(ref["log_r"]).sum() / n, k3(ref32["log_r"]).sum() / n
    lim = max(1e-5 * kl, kr * abs(kl32 - kl), _k3_floor(ref, ref32, logp_old, k) if first else 0.0)
    print("%s approx_kl %.6g vs %.6g: dev %.3g limit %.3g" % (tag, got[0], kl, abs(got[0] - kl), lim))
    if not abs(got[0] - kl) <= lim:
        fails.append((tag, "approx_kl", got[0], kl, lim))
    r64, r32 = np.exp(ref["log_r"]), np.exp(ref32["log_r"])
    win = np.where(big, np.maximum(1e-5, k * np.abs(r32 - r64)), 1e-5)
    near = int(((np.abs(r64 - 0.8) < win) | (np.abs(r64 - 1.2) < win)).sum())
    cnt = int(((r64 < 0.8) | (r64 > 1.2)).sum())
    if abs(got[1] - cnt) > near:
        fails.append((tag, "clip count", got[1], cnt, near))
    if head == 2:
        H, H32 = ref["H"].sum() / n, ref32["H"].sum() / n
        lim = max(1e-5 * abs(H), kr * abs(H32 - H))
        print("%s entropy %.8g vs %.8g: dev %.3g limit %.3g" % (tag, got[2], H, abs(got[2] - H), lim))
        if not abs(got[2] - H) <= lim:
            fails.append((tag, "entropy", got[2], H, lim))
    else:
        if not math.isnan(got[2]) and got[2] != 0.0:
            fails.append((tag, "entropy of a Gaussian pair", got[2]))
    ev, ev32 = _ev(ref["R"], ref["V"]), _ev(ref32["R"], ref32["V"])
    if math.isnan(ev):
        if not math.isnan(got[3]):
            fails.append((tag, "EV with Var(R) = 0", got[3]))
        return
    scale = max(abs(ev), abs(1 - ev))                # relative to the larger of the two terms of 1 - Var(R-V) / Var(R)
    lim = max(1e-5 * scale, kr * abs(ev32 - ev))
    print("%s explained variance %.8g vs %.8g: dev %.3g limit %.3g" % (tag, got[3], ev, abs(got[3] - ev), lim))
    if not abs(got[3] - ev) <= lim:
        fails.append((tag, "EV", got[3], ev, lim))


@pytest.mark.parametrize("case", ["full10", "mb3x3"])
def test_update_record_matches_fp64_restatement(mlp_mode, case):
    opts = dict(n_minibatches=3) if case == "mb3x3" else {}
    epochs = 10 if case == "full10" else 3
    algo = _algo(1024, seed=11, diagnostics=True, **opts)
    steps = _capture(algo)
    algo.update(epochs=epochs)
    torch.cuda.synchronize()
    r = algo.rollout
    T, M = r.T, r.M
    npc = lambda t: t.cpu().numpy()
    obs_c, rtg, act, logp = npc(r.obs_c), npc(r.rtg), npc(r.act), npc(r.logp)
    obs_d, rew_d, act_d, logp_d = npc(r.obs_d), npc(r.rew_d), npc(r.act_d), npc(r.logp_d)
    fails = []
    for w, pair in enumerate(("cross", "wait", "choice")):
        rec = algo.last_update_stats[pair]
        assert len(rec) == len(steps[w]) > 0, (pair, len(rec), len(steps[w]))
        for i, st in enumerate(steps[w]):
            cols = st["cols"]
            if w == 2:
                slots, x, R, a, lo = cols, obs_d[:, cols].T, rew_d[cols], act_d[cols], logp_d[cols]
            else:
                slots = (np.arange(T)[:, None] * M + cols[None, :]).reshape(-1)
                x, R, a, lo = obs_c[:, slots].T, rtg[slots], act[slots], logp[slots]
            assert rec["n"][i] == len(slots) == st["n"]
            got = (rec["approx_kl"][i], int(round(rec["clip_fraction"][i] * st["n"])), rec["entropy"][i], rec["explained_variance"][i])
            _compare(got, x, R, a, lo, st["a"], st["c"], 2 if w == 2 else 1, K32[mlp_mode], "mode %d %s %s step %d" % (mlp_mode, case, pair, i), fails,
                     first=(i == 0))
    assert not fails, fails


# per kernel, through the C ABI: widths, tile / grid boundaries, empty rank, ±1e3 rows
def _kernel_case(lay, D, head, seed, big_cols=False, mode=0):
    L = _lib()
    kp = L.mhppo_net_padded_in(D)
    rng = np.random.default_rng(seed)
    csd, asd = _net_sd(D, 1, 0, seed), _net_sd(D, 2 if head == 2 else 1, head, seed + 1)
    Q = lay["T"] * lay["K"]
    b = _draw_batch(rng, max(Q, 1), D, head, csd, asd, "mixed", DEFAULT_HEAD, big_cols) if Q else None
    S, idx, K, CN = lay["S"], lay["idx"], lay["K"], lay["CN"]
    if Q:
        x, rtg, act, logp = _scatter(lay, b["x"], D), _scatter(lay, b["rtg"]), _scatter(lay, b["act"]), _scatter(lay, b["logp"])
    else:
        x, rtg, act, logp = (torch.full(s, float("nan"), device="cuda") for s in ((D, S), (S,), (S,), (S,)))
    net_c, net_a = _pack(csd, D).cuda(), _pack(asd, D).cuda()
    n_glob = Q if Q else 100
    f0 = float((b["act"] == 0).sum()) / n_glob if Q else 0.0
    f1 = float((b["act"] == 1).sum()) / n_glob if Q else 0.0
    npar = L.mhppo_net_param_count(D)
    ws = torch.zeros(L.mhppo_update_workspace_bytes(D), dtype=torch.uint8, device="cuda")
    ip = None if idx is None else idx.data_ptr()
    out = {}
    for diag in (False, True):
        o = dict(V=torch.full((S,), float("nan"), device="cuda"), gc=torch.zeros(npar + 1, device="cuda"), ga=torch.zeros(npar + 1, device="cuda"),
                 st=torch.zeros(3, dtype=torch.float64, device="cuda"), lc=torch.zeros(1, dtype=torch.float64, device="cuda"),
                 la=torch.zeros(1, dtype=torch.float64, device="cuda"), rec=torch.zeros(10, dtype=torch.float64, device="cuda"))
        if diag:
            _check(L.mhppo_critic_grad_diag(D, x.data_ptr(), D, S, ip, K, CN, net_c.data_ptr(), rtg.data_ptr(), 1.0 / n_glob, o["gc"].data_ptr(),
                                            o["lc"].data_ptr(), o["V"].data_ptr(), o["st"].data_ptr(), o["rec"].data_ptr(), ws.data_ptr(), None))
            _check(L.mhppo_ppo_grad_diag(D, head, x.data_ptr(), D, S, ip, K, CN, net_a.data_ptr(), act.data_ptr(), logp.data_ptr(), rtg.data_ptr(),
                                         o["V"].data_ptr(), o["st"].data_ptr(), 1.0 / n_glob, f0, f1, 0.0, o["ga"].data_ptr(), o["la"].data_ptr(),
                                         o["ga"].data_ptr() + 4 * npar, o["rec"].data_ptr(), ws.data_ptr(), None))
        else:
            _check(L.mhppo_critic_grad_stats(D, x.data_ptr(), D, S, ip, K, CN, net_c.data_ptr(), rtg.data_ptr(), 1.0 / n_glob, o["gc"].data_ptr(),
                                             o["lc"].data_ptr(), o["V"].data_ptr(), o["st"].data_ptr(), ws.data_ptr(), None))
            _check(L.mhppo_ppo_grad_dev(D, head, x.data_ptr(), D, S, ip, K, CN, net_a.data_ptr(), act.data_ptr(), logp.data_ptr(), rtg.data_ptr(),
                                        o["V"].data_ptr(), o["st"].data_ptr(), 1.0 / n_glob, f0, f1, o["ga"].data_ptr(), o["la"].data_ptr(),
                                        ws.data_ptr(), None))
        torch.cuda.synchronize()
        out[diag] = {k: v.cpu() for k, v in o.items()}
    p, d = out[False], out[True]
    for k in ("V", "st", "lc", "la"):
        assert _bits_equal(p[k], d[k]), k
    assert _bits_equal(p["gc"][:npar], d["gc"][:npar]) and _bits_equal(p["ga"][:npar], d["ga"][:npar])
    rec = d["rec"].numpy()
    assert rec[0] == d["la"].item() and rec[1] == d["lc"].item() and rec[9] == 0.0
    assert np.float32(rec[2]) == d["ga"][npar].item()                      # the fp32 k3 slot
    if Q == 0:
        assert (rec == 0).all()
        return
    fails = []
    got = (rec[2] / Q, int(rec[3]), rec[4] / Q if head == 2 else float("nan"), None)
    Rv = b["rtg"].astype(np.float64)
    nvar = lambda s1, s2: s2 / Q - (s1 / Q) ** 2
    got = got[:3] + (1.0 - nvar(rec[5], rec[6]) / nvar(rec[7], rec[8]),)
    assert abs(rec[7] - Rv.sum()) <= 1e-12 * np.abs(Rv).sum() and abs(rec[8] - (Rv * Rv).sum()) <= 1e-12 * (Rv * Rv).sum()
    if head == 1:
        assert rec[4] == 0.0
    k = K32[mode] if big_cols else 2.0
    _compare(got, b["x"], b["rtg"], b["act"], b["logp"], asd, csd, head, k, "kernel D %d head %d Q %d%s" % (D, head, Q, " ±1e3" if big_cols else ""), fails)
    assert not fails, fails


@pytest.mark.parametrize("D", [13, 12, 18, 30, 42, 54])
def test_kernel_record_input_widths(mlp_mode, D):
    """13 = the cross / wait nets (both heads), 12 and 18 / 30 / 42 / 54 = choice widths of the older drivers and nb_lines 1-4."""
    G, _ = _grid()
    rng = np.random.default_rng(D)
    for head in ((1, 2) if D == 13 else (2,)):
        _kernel_case(_layout(1, 256 * G + 3, 256 * G + 8, "list", rng), D, head, 500 + 10 * D + head, mode=mlp_mode)


@pytest.mark.parametrize("qn", ["0", "128G-1", "128G+1", "256G-1", "256G+1"])
def test_kernel_record_boundaries(mlp_mode, qn):
    """Tile and grid boundaries of the 128-sample (tensor-core) and 256-sample (FFMA) tiles; Q = 0 is a rank without samples."""
    G, _ = _grid()
    Q = {"0": 0, "128G-1": 128 * G - 1, "128G+1": 128 * G + 1, "256G-1": 256 * G - 1, "256G+1": 256 * G + 1}[qn]
    rng = np.random.default_rng(Q)
    lay = _layout(1, Q, Q + 7, "empty" if Q == 0 else "list", rng)
    for head, D in ((1, 13), (2, 30)):
        _kernel_case(lay, D, head, 600 + Q % 1000 + head, mode=mlp_mode)


@pytest.mark.parametrize("head,D", [(1, 13), (2, 18), (2, 30)])
def test_kernel_record_placeholder_rows(mlp_mode, head, D):
    G, _ = _grid()
    rng = np.random.default_rng(40 + D)
    Q = 128 * G + 77
    _kernel_case(_layout(2, Q // 2, Q // 2 + 9, "list", rng), D, head, 700 + D, big_cols=True, mode=mlp_mode)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the target-KL halt

def _snapshots(algo):
    """Wrap _step_pair: each pair's (flat, m, v) of actor and critic after every launched step."""
    snaps = {id(a): [] for _, a, _ in algo._pair_nets()}
    sp = algo._step_pair

    def wrap(actor, critic, oa, oc, *a):
        sp(actor, critic, oa, oc, *a)
        snaps[id(actor)].append([t.clone() for net in (actor, critic) for t in (net.flat, net.m, net.v)])
    algo._step_pair = wrap
    return snaps


@pytest.mark.parametrize("case", ["full", "B4"])
def test_target_kl_halts_where_the_kl_first_exceeds(mlp_mode, case):
    opts = dict(n_minibatches=4) if case == "B4" else {}
    base = _algo(2048, diagnostics=True, **opts)
    init = {p: [t.clone() for net in (a, c) for t in (net.flat, net.m, net.v)] + [a.step] for p, a, c in base._pair_nets()}
    snaps = _snapshots(base)
    base.update(epochs=4)
    torch.cuda.synchronize()
    st = base.last_update_stats
    choice = None
    for p in ("cross", "wait", "choice"):
        kl = st[p]["approx_kl"]
        for j in range(1, len(kl)):
            if kl[j] > kl[:j].max():
                choice = (p, j, 0.5 * (kl[j] + kl[:j].max()))
                break
        if choice:
            break
    assert choice is not None
    P, j, lim = choice
    delta = lim / 1.5
    halted = _algo(2048, target_kl=delta, **opts)
    halted.update(epochs=4)
    torch.cuda.synchronize()
    for p, a, c in halted._pair_nets():
        kl = st[p]["approx_kl"]
        h = int(np.argmax(kl > lim)) if (kl > lim).any() else len(kl)
        if p == P:
            assert h == j
        tk = halted.last_update_stats[p]["taken"]
        assert tk.tolist() == [True] * h + [False] * (len(kl) - h), (p, tk, h)
        want = init[p][:6] if h == 0 else snaps[id(getattr(base, "actor_net_" + p))][h - 1]
        got = [t for net in (a, c) for t in (net.flat, net.m, net.v)]
        assert all(_bits_equal(x, y) for x, y in zip(got, want)), p
        assert a.step == c.step == init[p][6] + h
        # the records of the steps both runs took are the same bits
        for f in ("approx_kl", "clip_fraction", "explained_variance", "actor_loss", "critic_loss"):
            assert np.array_equal(halted.last_update_stats[p][f][:h], st[p][f][:h])
    # the next update starts from the settled step counts and a cleared halt
    halted.rollout.iterations_rand(halted.actor_net_cross, halted.actor_net_wait, halted.actor_net_choice)
    halted.update(epochs=1)
    torch.cuda.synchronize()
    assert all(len(v) for v in halted.last_update_stats.values())


# ---------------------------------------------------------------------------------------------------------------------
# 4. determinism, 5. two ranks

def test_records_are_deterministic(mlp_mode):
    a, b = (_algo(2048, n_minibatches=4, gae_lambda=0.95, entropy_coef=0.01, diagnostics=True) for _ in range(2))
    a.update(epochs=3)
    b.update(epochs=3)
    torch.cuda.synchronize()
    for p in a.last_update_stats:
        assert a.last_update_stats[p].tobytes() == b.last_update_stats[p].tobytes(), p


def test_train_appends_diagnostics(mlp_mode):
    algo = _algo(512, nb=(1, 1, 1), diagnostics=True)
    algo.train(2, save_traces=False)
    assert len(algo.ep_diagnostics) == 2
    for it in algo.ep_diagnostics:
        assert set(it) == {"cross", "wait", "choice"}
        for p, d in it.items():
            assert d["steps_taken"] == d["steps_launched"]


def test_two_rank_record_equals_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29527", os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "OK" in r.stdout


def _dist_main():
    """Two ranks of N/2 envs against one rank of N envs, diagnostics and a target_kl that halts: the same records on both ranks,
    the same halt decisions, and the record within the bars of tests/dist_ppo_check.py (1e-4 relative) of the one-rank run."""
    import torch.distributed as dist
    import mhppo_b200
    from mhppo_b200 import ppo
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    N = 4096
    n = N // world

    def run(N, env_id0, use_dist, **opts):
        ppo.set_distributed(use_dist)
        env = mhppo_b200.VecCrosswalkEnv("coop_scalable", N, nb_car=4, nb_ped=3, nb_lines=2, seed=77, env_id0=env_id0, device=dev)
        torch.manual_seed(0 if not use_dist else 1000 * rank)
        algo = mhppo_b200.Algo_PPO(mhppo_b200.Model_PPO, env, num_states_c=13, num_states_d=30, num_actions=1, mean=-1.0, std=3.0,
                                   nb_cars=4, dt=0.3, **opts)
        algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        algo.update(epochs=4)
        torch.cuda.synchronize()
        return algo
    whole = run(N, 0, False, diagnostics=True)
    kl = whole.last_update_stats["cross"]["approx_kl"]
    delta = (0.5 * (kl[1] + kl[0]) if kl[1] > kl[0] else 2 * kl.max() + 1e-12) / 1.5
    sharded = run(n, rank * n, True, target_kl=delta)
    whole = run(N, 0, False, target_kl=delta)
    worst = 0.0
    for p in ("cross", "wait", "choice"):
        a, b = sharded.last_update_stats[p], whole.last_update_stats[p]
        assert a["taken"].tolist() == b["taken"].tolist(), p
        for f in ("approx_kl", "clip_fraction", "explained_variance", "actor_loss", "critic_loss"):
            d = np.abs(a[f] - b[f]) / np.maximum(np.abs(b[f]), 1e-12)
            worst = max(worst, float(np.nanmax(d)) if len(d) else 0.0)
        t = torch.as_tensor(a.view(np.uint8).copy(), device=dev)
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        assert all(torch.equal(g[0], x) for x in g), "ranks disagree on the record"
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("two-rank diagnostics world=%d: same records on every rank, same halts, max relative difference to one rank %.3e" % (world, t.item()))
    assert t.item() < 1e-4, t.item()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    _dist_main()
