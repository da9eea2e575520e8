"""Per-net gradient-norm clipping on the GPU (Algo_PPO(max_grad_norm=g), mhppo_adam2_clip): the kernel alone against the float64
restatement of tests/test_grad_clip.py at sizes around every warp and CTA boundary, bit-identity with mhppo_adam2 /
mhppo_adam2_halt whenever nothing is clipped, max_grad_norm=inf against None over whole updates, real clipped steps against the
restatement from the state before each step, the padded gradient slots, and the per-step norm records.

Bars: the norm within 1e-12 relative of the float64 norm of the fp32 gradient; p, m and v within 8 fp32 roundings of the
magnitudes that enter each (the kernel forms coef and the step in fp32; the restatement takes the fp32 values of beta1, beta2, eps
and lr that the kernel receives)."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_grad_clip import clip_coef, clipped_adam64  # noqa: E402
from test_ppo_diagnostics_gpu import _algo, _state, _same_state, mlp_mode  # noqa: E402,F401
from test_update_kernels_gpu import _bits_equal  # noqa: E402

pytestmark = pytest.mark.gpu
EPS32 = 2.0 ** -24
EINVAL = -1
SIZES = [1, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 4868, 5380, 6148]
HP = [(1e-3, 3), (3e-4, 1)]                       # (lr, step) of net 0 (actor) and net 1 (critic)


def _lib():
    import mhppo_b200
    return mhppo_b200.lib()


# ---------------------------------------------------------------------------------------------------------------------
# float64 restatement and its bars

def _close_to_restatement(new, old, g, lr, step, max_norm, tag):
    """new / old: dicts of p, m, v (numpy float32) after / before one net's step; g its fp32 gradient."""
    f = lambda a: np.asarray(a, np.float64)
    b1, b2, eps, lr = (float(np.float32(x)) for x in (0.9, 0.999, 1e-8, lr))          # the constants as the kernel receives them
    p64, m64, v64, norm = clipped_adam64(f(old["p"]), f(old["m"]), f(old["v"]), f(g), step, lr, max_norm, b1, b2, eps)
    gi = np.abs(f(g)) * clip_coef(norm, max_norm)
    sm = b1 * np.abs(f(old["m"])) + (1.0 - b1) * gi
    sv = b2 * f(old["v"]) + (1.0 - b2) * gi * gi
    den = np.sqrt(v64) / math.sqrt(1.0 - b2 ** step) + eps
    sp = np.abs(p64) + lr / (1.0 - b1 ** step) * (sm + np.abs(m64)) / den
    for name, got, ref, scale in (("m", new["m"], m64, sm), ("v", new["v"], v64, sv), ("p", new["p"], p64, sp)):
        err = np.abs(f(got) - ref)
        assert (err <= 8 * EPS32 * scale + 1e-30).all(), (tag, name, float((err / (scale + 1e-30)).max()))
    return norm


# ---------------------------------------------------------------------------------------------------------------------
# 1. the kernel alone

def _nets(n0, n1, seed, gscale=(1.0, 0.3)):
    rng = np.random.default_rng(seed)
    mk = lambda n, s: dict(p=rng.normal(size=n), g=rng.normal(size=n) * s, m=rng.normal(size=n) * 1e-2, v=rng.random(n) * 1e-3)
    return [{k: v.astype(np.float32) for k, v in mk(n, s).items()} for n, s in ((n0, gscale[0]), (n1, gscale[1]))]


def _call(fn, nets, *extra):
    """Runs fn (an mhppo_adam2* entry) on device copies of nets; returns (return code, the two nets after the call)."""
    d = [{k: torch.from_numpy(v).cuda() for k, v in x.items()} for x in nets]
    args = []
    for (lr, step), x in zip(HP, d):
        args += [x["p"].data_ptr(), x["g"].data_ptr(), x["m"].data_ptr(), x["v"].data_ptr(), x["p"].numel(), lr, step]
    rc = fn(*args, 0.9, 0.999, 1e-8, *extra, None)
    torch.cuda.synchronize()
    return rc, [{k: v.cpu().numpy() for k, v in x.items()} for x in d]


def _clip(nets, max_norm, halt=None):
    """mhppo_adam2_clip; halt = (kl_sum, kl_limit, halt flag) or None.  Returns (nets after, norms, halt flag, record row)."""
    L = _lib()
    norms = torch.full((2,), float("nan"), dtype=torch.float64, device="cuda")
    if halt is None:
        rc, out = _call(L.mhppo_adam2_clip, nets, max_norm, norms.data_ptr(), None, 0.0, None, None)
        assert rc == 0
        return out, norms.cpu().numpy(), None, None
    kl = torch.tensor([halt[0]], dtype=torch.float32, device="cuda")
    flag = torch.tensor([halt[2]], dtype=torch.int32, device="cuda")
    row = torch.zeros(10, dtype=torch.float64, device="cuda")
    rc, out = _call(L.mhppo_adam2_clip, nets, max_norm, norms.data_ptr(), kl.data_ptr(), halt[1], flag.data_ptr(), row.data_ptr())
    assert rc == 0
    return out, norms.cpu().numpy(), int(flag.item()), row.cpu().numpy()


def _same_bits(a, b):
    return all(np.array_equal(a[k].view(np.int32), b[k].view(np.int32)) for k in ("p", "m", "v", "g"))


@pytest.mark.parametrize("i", range(len(SIZES)))
def test_kernel_matches_restatement(i):
    n0, n1 = SIZES[i], SIZES[(i + 5) % len(SIZES)]
    nets = _nets(n0, n1, 100 + i)
    norms64 = [math.sqrt(float(np.dot(x["g"].astype(np.float64), x["g"].astype(np.float64)))) for x in nets]
    _, plain = _call(_lib().mhppo_adam2, nets)
    lo, hi = min(norms64), max(norms64)
    for max_norm in (math.inf, 1e30, 2.0 * hi, math.sqrt(lo * hi), 0.5 * lo):
        out, norms, _, _ = _clip(nets, max_norm)
        for y in range(2):
            tag = "n %d / %d net %d max_norm %g" % (n0, n1, y, max_norm)
            assert abs(norms[y] - norms64[y]) <= 1e-12 * norms64[y], (tag, norms[y], norms64[y])
            assert np.array_equal(out[y]["g"].view(np.int32), nets[y]["g"].view(np.int32)), tag          # g is not written
            _close_to_restatement(out[y], nets[y], nets[y]["g"], HP[y][0], HP[y][1], max_norm, tag)
            if clip_coef(norms64[y], max_norm) == 1.0:
                assert _same_bits(out[y], plain[y]), tag                                                # unclipped = mhppo_adam2
        again, norms2, _, _ = _clip(nets, max_norm)
        assert all(_same_bits(a, b) for a, b in zip(out, again)) and np.array_equal(norms, norms2)     # repeatable bit for bit
    # a zero gradient: norm 0, coef 1
    z = [dict(x, g=np.zeros_like(x["g"])) for x in nets]
    out, norms, _, _ = _clip(z, 0.5)
    _, plain_z = _call(_lib().mhppo_adam2, z)
    assert (norms == 0.0).all() and all(_same_bits(a, b) for a, b in zip(out, plain_z))


@pytest.mark.parametrize("sizes", [(4868, 4868), (5380, 4868), (6148, 33)])
def test_kernel_halting_form(sizes):
    L = _lib()
    nets = _nets(*sizes, 7)
    norms64 = [math.sqrt(float(np.dot(x["g"].astype(np.float64), x["g"].astype(np.float64)))) for x in nets]

    def halt_ref(kl, limit, flag):
        k = torch.tensor([kl], dtype=torch.float32, device="cuda")
        f = torch.tensor([flag], dtype=torch.int32, device="cuda")
        row = torch.zeros(10, dtype=torch.float64, device="cuda")
        rc, out = _call(L.mhppo_adam2_halt, nets, k.data_ptr(), limit, f.data_ptr(), row.data_ptr())
        assert rc == 0
        return out, int(f.item()), row.cpu().numpy()
    # taken, nothing clipped: mhppo_adam2_halt bit for bit, taken = 1
    for max_norm in (math.inf, 2.0 * max(norms64)):
        out, norms, flag, row = _clip(nets, max_norm, (1.0, 2.0, 0))
        ref, rflag, rrow = halt_ref(1.0, 2.0, 0)
        assert all(_same_bits(a, b) for a, b in zip(out, ref)) and flag == rflag == 0 and row[9] == rrow[9] == 1.0
        assert all(abs(norms[y] - norms64[y]) <= 1e-12 * norms64[y] for y in range(2))
    # taken and clipped
    out, norms, flag, row = _clip(nets, 0.5 * min(norms64), (1.0, 2.0, 0))
    assert flag == 0 and row[9] == 1.0
    for y in range(2):
        _close_to_restatement(out[y], nets[y], nets[y]["g"], HP[y][0], HP[y][1], 0.5 * min(norms64), "halt form net %d" % y)
    # halted by the KL, or by an earlier step: nothing moves, the norms are still reported
    for kl, flag0 in ((3.0, 0), (1.0, 1)):
        out, norms, flag, row = _clip(nets, 0.5 * min(norms64), (kl, 2.0, flag0))
        assert flag == 1 and row[9] == 0.0
        assert all(_same_bits(a, b) for a, b in zip(out, nets))
        assert all(abs(norms[y] - norms64[y]) <= 1e-12 * norms64[y] for y in range(2))


def test_kernel_non_finite_gradient_takes_the_unclipped_step():
    L = _lib()
    nets = _nets(4868, 5380, 9)
    nets[0]["g"][17] = np.inf
    nets[1]["g"][4000] = np.nan
    _, plain = _call(L.mhppo_adam2, nets)
    with np.errstate(invalid="ignore"):
        out, norms, _, _ = _clip(nets, 0.5)
    assert math.isinf(norms[0]) and math.isnan(norms[1])
    for a, b in zip(out, plain):
        for k in ("p", "m", "v"):
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_kernel_bad_arguments():
    L = _lib()
    nets = _nets(64, 64, 1)
    kl = torch.zeros(1, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    row = torch.zeros(10, dtype=torch.float64, device="cuda")
    for max_norm in (math.nan, 0.0, -0.5, -math.inf):
        assert _call(L.mhppo_adam2_clip, nets, max_norm, None, None, 0.0, None, None)[0] == EINVAL, max_norm
    for ptrs in ((kl.data_ptr(), None, None), (None, flag.data_ptr(), None), (None, None, row.data_ptr()),
                 (kl.data_ptr(), flag.data_ptr(), None), (None, flag.data_ptr(), row.data_ptr())):
        assert _call(L.mhppo_adam2_clip, nets, 0.5, None, ptrs[0], 1.0, ptrs[1], ptrs[2])[0] == EINVAL, ptrs
    assert _call(L.mhppo_adam2_clip, nets, 0.5, None, kl.data_ptr(), math.nan, flag.data_ptr(), row.data_ptr())[0] == EINVAL
    empty = [nets[0], {k: v[:0] for k, v in nets[1].items()}]                                         # n1 = 0
    assert _call(L.mhppo_adam2_clip, empty, 0.5, None, None, 0.0, None, None)[0] == EINVAL


# ---------------------------------------------------------------------------------------------------------------------
# 2. max_grad_norm = inf changes no bit of an update

SETTINGS = {"full": {}, "B4": dict(n_minibatches=4), "gae_entropy": dict(gae_lambda=0.95, entropy_coef=0.01), "kl_never": dict(target_kl=1e9)}


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_inf_leaves_the_update_bit_identical(mlp_mode, setting):
    opts = SETTINGS[setting]
    ref = _algo(2048, **opts)
    ref.update()
    torch.cuda.synchronize()
    a = _algo(2048, max_grad_norm=math.inf, **opts)
    a.update()
    torch.cuda.synchronize()
    assert _same_state(_state(ref), _state(a))
    assert _bits_equal(ref._loss, a._loss)
    if "target_kl" in opts:
        for p in ref.last_update_stats:
            assert ref.last_update_stats[p].tobytes() == a.last_update_stats[p].tobytes(), p
    for p, arr in a.last_grad_norms.items():
        assert len(arr) > 0 and np.isfinite(arr["actor_grad_norm"]).all() and (arr["critic_grad_norm"] > 0).all(), p
        if "target_kl" in opts:
            assert len(arr) == len(a.last_update_stats[p])


# ---------------------------------------------------------------------------------------------------------------------
# 3. real clipped steps against the restatement, and the padded gradient slots

def _pad_slots(net):
    """Flat indices of the padded slots: W1^T rows n_in .. KP, the W4^T columns and b4 entries n_out .. 4."""
    kp, n_in, n_out = net.kp, net.n_in, net.n_out
    w4 = kp * 32 + 32 + 32 * 64 + 64 + 64 * 32 + 32
    idx = list(range(n_in * 32, kp * 32)) + [w4 + k * 4 + j for k in range(32) for j in range(n_out, 4)] + \
        [w4 + 128 + j for j in range(n_out, 4)]
    assert len(idx) == (kp - n_in) * 32 + 33 * (4 - n_out)
    return torch.tensor(idx, dtype=torch.long, device=net.flat.device)


@pytest.mark.parametrize("nb", [(4, 3, 2), (4, 3, 4)], ids=["kp16_32", "kp16_56"])
def test_clipped_steps_match_restatement(mlp_mode, nb):
    G = 1e-6
    algo = _algo(1024, seed=5, nb=nb, max_grad_norm=G)
    steps = {"cross": [], "wait": [], "choice": []}
    names = {id(a): p for p, a, _ in algo._pair_nets()}
    sp = algo._step_pair

    def wrap(actor, critic, oa, oc, *a):
        before = [dict(p=n.flat.cpu().numpy(), m=n.m.cpu().numpy(), v=n.v.cpu().numpy(), step=n.step) for n in (actor, critic)]
        sp(actor, critic, oa, oc, *a)
        after = [dict(p=n.flat.cpu().numpy(), m=n.m.cpu().numpy(), v=n.v.cpu().numpy(), g=n.grad.cpu().numpy()) for n in (actor, critic)]
        pads = [bool((n.grad[_pad_slots(n)] == 0).all()) for n in (actor, critic)]
        steps[names[id(actor)]].append((before, after, (oa.lr, oc.lr), pads))
    algo._step_pair = wrap
    algo.update(epochs=2)
    torch.cuda.synchronize()
    kps = set()
    for p, a, c in algo._pair_nets():
        kps |= {a.kp, c.kp}
        rec = algo.last_grad_norms[p]
        assert len(rec) == len(steps[p]) > 0, p
        for j, (before, after, lrs, pads) in enumerate(steps[p]):
            assert all(pads), (p, j, "padded gradient slots not 0")
            if p == "wait":
                continue
            for y, field in enumerate(("actor_grad_norm", "critic_grad_norm")):
                tag = "mode %d %s step %d net %d" % (mlp_mode, p, j, y)
                norm = _close_to_restatement(after[y], before[y], after[y]["g"], lrs[y], before[y]["step"] + 1, G, tag)
                assert abs(rec[field][j] - norm) <= 1e-12 * norm, (tag, rec[field][j], norm)
                if nb == (4, 3, 2):
                    assert clip_coef(norm, G) < 1.0, (tag, norm)
    assert kps == ({16, 32} if nb == (4, 3, 2) else {16, 56})


# ---------------------------------------------------------------------------------------------------------------------
# 4. bookkeeping

def test_norm_records_line_up_with_the_diagnostics(mlp_mode):
    a = _algo(2048, n_minibatches=3, diagnostics=True, max_grad_norm=0.5)
    a.update(epochs=3)
    torch.cuda.synchronize()
    for p in ("cross", "wait", "choice"):
        g, d = a.last_grad_norms[p], a.last_update_stats[p]
        assert len(g) == len(d) > 0, p
        assert np.array_equal(g["epoch"], d["epoch"]) and np.array_equal(g["minibatch"], d["minibatch"]), p
    # without diagnostics: one entry per launched step, in launch order
    b = _algo(2048, n_minibatches=3, max_grad_norm=0.5)
    launched = {p: 0 for p in ("cross", "wait", "choice")}
    names = {id(x): p for p, x, _ in b._pair_nets()}
    sp = b._step_pair

    def count(actor, *args):
        launched[names[id(actor)]] += 1
        sp(actor, *args)
    b._step_pair = count
    b.update(epochs=3)
    torch.cuda.synchronize()
    for p in launched:
        g = b.last_grad_norms[p]
        assert len(g) == launched[p] > 0, p
        assert np.array_equal(g["epoch"], a.last_grad_norms[p]["epoch"]) and np.array_equal(g["minibatch"], a.last_grad_norms[p]["minibatch"])
        assert np.array_equal(g["actor_grad_norm"], a.last_grad_norms[p]["actor_grad_norm"]), p       # diagnostics change no bit
    # outside update(): the step clips, nothing is recorded
    before = {p: v.copy() for p, v in b.last_grad_norms.items()}
    assert b.train_model_c(b.actor_net_cross, b.critic_net_cross, b.optimizer_actor_cross, b.optimizer_critic_cross, 0)
    torch.cuda.synchronize()
    assert all(np.array_equal(before[p], b.last_grad_norms[p]) for p in before)


def test_halted_steps_still_record_norms(mlp_mode):
    """Every pair halts at its first step (target_kl far below the first step's approx. KL on a rollout the weights have moved
    away from): the norms are still recorded, equal to those of the same step in a twin run that takes it, and no weight moves."""
    twin = _algo(2048, target_kl=1e9, max_grad_norm=0.5)
    twin.update()
    twin.update()
    torch.cuda.synchronize()
    first_kl = min(float(twin.last_update_stats[p]["approx_kl"][0]) for p in twin.last_update_stats)
    assert first_kl > 0
    a = _algo(2048, target_kl=1e9, max_grad_norm=0.5)
    a.update()
    a.target_kl = min(1e-3, first_kl / 3.0)
    torch.cuda.synchronize()
    s0 = _state(a)
    a.update()
    torch.cuda.synchronize()
    assert _same_state(s0, _state(a))
    for p in ("cross", "wait", "choice"):
        st, g = a.last_update_stats[p], a.last_grad_norms[p]
        assert len(g) == len(st) > 0 and not st["taken"].any(), p
        assert np.isfinite(g["actor_grad_norm"]).all() and (g["critic_grad_norm"] > 0).all(), p
        # the parameters never move, so every launched step has the first step's gradient
        t = twin.last_grad_norms[p]
        assert (g["actor_grad_norm"] == t["actor_grad_norm"][0]).all() and (g["critic_grad_norm"] == t["critic_grad_norm"][0]).all(), p


def test_train_appends_grad_norms(mlp_mode):
    algo = _algo(512, nb=(1, 1, 1), max_grad_norm=0.5)
    algo.train(2, save_traces=False)
    assert len(algo.ep_grad_norms) == 2
    for it in algo.ep_grad_norms:
        assert set(it) == {"cross", "wait", "choice"}
