"""Learning-rate schedules on the GPU (Algo_PPO(lr_schedule="linear" | "adaptive"), mhppo_adam2_sched): the kernel alone against
the restated rule of tests/test_lr_schedule.py at sizes around every warp and CTA boundary, bit-identity with mhppo_adam2 /
mhppo_adam2_clip whenever the lr does not change, the halt, "linear" against a default Algo_PPO whose lrs are set by hand, and
"adaptive" updates: every step's lr against the rule driven by that step's recorded approx. KL, the weights against the float64
restatement of tests/test_minibatch_gpu.py fed the recorded lrs, clipping and the target-KL halt on top, the lr state across
updates, the launch count of the default update and (two GPUs) two ranks against one.

Bars: lrs exactly, except at a step whose fp64 record KL lies within 1e-6 relative of 2 delta or delta / 2 (the kernel decides on
the fp32 all-reduced k3 sum): such a step may go either way, and the tests count and print them.  Weights: the bars of
tests/test_minibatch_gpu.py for the same mode and pair; a clipped step: the bars of tests/test_grad_clip_gpu.py."""
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

from test_lr_schedule import adaptive_lr, linear_lr  # noqa: E402
from test_grad_clip_gpu import SIZES, HP, _nets, _call, _same_bits, _close_to_restatement  # noqa: E402
from test_ppo_diagnostics_gpu import _algo, _state, _same_state, mlp_mode  # noqa: E402,F401
from test_minibatch_gpu import _reference_mb_update, _sd64  # noqa: E402
from test_update_kernels_gpu import _pack  # noqa: E402

pytestmark = pytest.mark.gpu
EINVAL = -1
DELTA = 0.01
PAIRS = ("cross", "wait", "choice")


def _lib():
    import mhppo_b200
    return mhppo_b200.lib()


# ---------------------------------------------------------------------------------------------------------------------
# 1. the kernel alone

def _sched(nets, lr_state, kl_sum, n, delta, max_norm=math.inf, halt=None):
    """mhppo_adam2_sched with the lr state lr_state (two fp32 values) and the fp32 KL slot kl_sum; halt = (kl_limit, flag) or None
    (the halt reads the same slot).  Returns (nets after, lr state after, lrs row, norms, halt flag, record row)."""
    L = _lib()
    lr = torch.tensor(lr_state, dtype=torch.float32, device="cuda")
    kl = torch.tensor([kl_sum], dtype=torch.float32, device="cuda")
    lrs = torch.full((2,), math.nan, dtype=torch.float64, device="cuda")
    norms = torch.full((2,), math.nan, dtype=torch.float64, device="cuda")
    flag = torch.tensor([0 if halt is None else halt[1]], dtype=torch.int32, device="cuda")
    row = torch.zeros(10, dtype=torch.float64, device="cuda")
    h = (None, 0.0, None, None) if halt is None else (kl.data_ptr(), halt[0], flag.data_ptr(), row.data_ptr())
    rc, out = _call(L.mhppo_adam2_sched, nets, max_norm, norms.data_ptr(), *h, lr.data_ptr(), kl.data_ptr(), float(n), float(delta),
                    lrs.data_ptr())
    assert rc == 0
    return out, lr.cpu().numpy(), lrs.cpu().numpy(), norms.cpu().numpy(), int(flag.item()), row.cpu().numpy()


def _adam2_with(nets, lrs):
    """mhppo_adam2 with the two lrs in place of HP's (same steps)."""
    L = _lib()
    d = [{k: torch.from_numpy(v).cuda() for k, v in x.items()} for x in nets]
    args = []
    for (_, step), lr, x in zip(HP, lrs, d):
        args += [x["p"].data_ptr(), x["g"].data_ptr(), x["m"].data_ptr(), x["v"].data_ptr(), x["p"].numel(), float(lr), step]
    assert L.mhppo_adam2(*args, 0.9, 0.999, 1e-8, None) == 0
    torch.cuda.synchronize()
    return [{k: v.cpu().numpy() for k, v in x.items()} for x in d]


def _clip_with(nets, max_norm):
    L = _lib()
    norms = torch.zeros(2, dtype=torch.float64, device="cuda")
    rc, out = _call(L.mhppo_adam2_clip, nets, max_norm, norms.data_ptr(), None, 0.0, None, None)
    assert rc == 0
    return out, norms.cpu().numpy()


@pytest.mark.parametrize("i", range(len(SIZES)))
def test_kernel_matches_restatement(i):
    n0, n1 = SIZES[i], SIZES[(i + 5) % len(SIZES)]
    nets = _nets(n0, n1, 200 + i)
    lr0 = [float(np.float32(lr)) for lr, _ in HP]
    n = 1000.0 + 37 * i
    # a KL slot of exactly delta * n: the lr stays, the step is mhppo_adam2's (mhppo_adam2_clip's) bit for bit
    norms64 = [math.sqrt(float(np.dot(x["g"].astype(np.float64), x["g"].astype(np.float64)))) for x in nets]
    plain = _adam2_with(nets, lr0)
    for max_norm in (math.inf, 0.5 * min(norms64)):
        out, lr, lrs, norms, _, _ = _sched(nets, lr0, DELTA * n, n, DELTA, max_norm)
        ref, ref_norms = _clip_with(nets, max_norm)
        assert lr.tolist() == lr0 and lrs.tolist() == lr0, (max_norm, lr, lrs)
        assert all(_same_bits(a, b) for a, b in zip(out, ref)), max_norm
        assert np.array_equal(norms, ref_norms)
        if max_norm == math.inf:
            assert all(_same_bits(a, b) for a, b in zip(out, plain))
    # decisions: increase, decrease, both clamps, kl = 0 and NaN give the restated lr, and the step is mhppo_adam2's at that lr
    cases = [(lr0, 0.25 * DELTA * n), (lr0, 4.0 * DELTA * n), ([1.2e-5, 1e-5], 4.0 * DELTA * n), ([8e-3, 1e-2], 0.1 * DELTA * n),
             (lr0, 0.0), (lr0, math.nan), (lr0, math.inf), (lr0, -1.0)]
    for state, kl_sum in cases:
        state = [float(np.float32(x)) for x in state]
        out, lr, lrs, _, _, _ = _sched(nets, state, kl_sum, n, DELTA)
        kl = float(np.float32(kl_sum)) / n
        want = [adaptive_lr(x, kl, DELTA) for x in state]
        tag = (n0, n1, state, kl_sum)
        assert lr.tolist() == want and lrs.tolist() == want, (tag, lr, lrs, want)
        assert all(_same_bits(a, b) for a, b in zip(out, _adam2_with(nets, want))), tag
    # with the halt: a set flag, or a KL over the limit, leaves p, m, v, the lr state and the lr row untouched
    for flag0, limit in ((1, 1e30), (0, 0.5 * DELTA * n)):
        out, lr, lrs, _, flag, row = _sched(nets, lr0, DELTA * n, n, DELTA, halt=(limit, flag0))
        assert flag == 1 and row[9] == 0.0 and lr.tolist() == lr0 and np.isnan(lrs).all()
        assert all(_same_bits(a, b) for a, b in zip(out, nets))
    out, lr, lrs, _, flag, row = _sched(nets, lr0, 4.0 * DELTA * n, n, DELTA, halt=(1e30, 0))     # taken: adapts as without the halt
    want = [adaptive_lr(x, float(np.float32(4.0 * DELTA * n)) / n, DELTA) for x in lr0]
    assert flag == 0 and row[9] == 1.0 and lr.tolist() == want and lrs.tolist() == want
    assert all(_same_bits(a, b) for a, b in zip(out, _adam2_with(nets, want)))


def test_kernel_bad_arguments():
    L = _lib()
    nets = _nets(64, 64, 1)
    lr = torch.full((2,), 1e-3, device="cuda")
    kl = torch.zeros(1, device="cuda")
    base = (math.inf, None, None, 0.0, None, None)
    assert _call(L.mhppo_adam2_sched, nets, *base, lr.data_ptr(), kl.data_ptr(), 10.0, 0.01, None)[0] == 0
    for lrp, klp, n, d in ((None, kl.data_ptr(), 10.0, 0.01), (lr.data_ptr(), None, 10.0, 0.01), (lr.data_ptr(), kl.data_ptr(), 10.0, 0.0),
                           (lr.data_ptr(), kl.data_ptr(), 10.0, -0.01), (lr.data_ptr(), kl.data_ptr(), 10.0, math.nan),
                           (lr.data_ptr(), kl.data_ptr(), 0.0, 0.01), (lr.data_ptr(), kl.data_ptr(), math.nan, 0.01)):
        assert _call(L.mhppo_adam2_sched, nets, *base, lrp, klp, n, d, None)[0] == EINVAL, (lrp, klp, n, d)
    assert _call(L.mhppo_adam2_sched, nets, 0.0, *base[1:], lr.data_ptr(), kl.data_ptr(), 10.0, 0.01, None)[0] == EINVAL
    assert _call(L.mhppo_adam2_sched, nets, math.inf, None, kl.data_ptr(), 1.0, None, None, lr.data_ptr(), kl.data_ptr(), 10.0, 0.01,
                 None)[0] == EINVAL
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 2. "linear": a default Algo_PPO with the six lrs set by hand, bit for bit

def _opts(algo):
    return [o for _, pair in algo._pair_optimizers() for o in pair]


def test_linear_equals_lrs_set_by_hand(mlp_mode):
    K = 2
    a = _algo(2048, lr_schedule="linear", lr_anneal_iterations=K)
    b = _algo(2048)
    lr0 = [o.lr for o in _opts(b)]
    for it in range(3):                                  # k = 0, 1, 2: fractions 1, 1/2, 0
        for o, l0 in zip(_opts(b), lr0):
            o.lr = linear_lr(l0, b.total_loop, K)
        a.train(1, save_traces=False)
        b.train(1, save_traces=False)
        torch.cuda.synchronize()
        assert _same_state(_state(a), _state(b)), it
        assert [o.lr for o in _opts(a)] == [o.lr for o in _opts(b)], it
        for p, (oa, oc) in a._pair_optimizers():
            rec = a.last_lrs[p]
            assert len(rec) == 10 and (rec["actor_lr"] == float(np.float32(oa.lr))).all() and (rec["critic_lr"] == float(np.float32(oc.lr))).all()
    assert all(o.lr == 0.0 for o in _opts(a)) and len(a.ep_lrs) == 3


def test_default_update_launches(mlp_mode):
    import mhppo_b200 as mh
    counts = {}
    for name, opts in (("none", {}), ("linear", dict(lr_schedule="linear", lr_anneal_iterations=10)), ("diagnostics", dict(diagnostics=True)),
                       ("adaptive", dict(lr_schedule="adaptive", desired_kl=DELTA))):
        a = _algo(2048, **opts)
        n0 = mh.launch_count()
        a.update()
        torch.cuda.synchronize()
        counts[name] = mh.launch_count() - n0
    print("launches per update at 4/3/2:", counts)
    assert counts["none"] == counts["linear"] == 151
    assert counts["adaptive"] == counts["diagnostics"]


# ---------------------------------------------------------------------------------------------------------------------
# 3. "adaptive" updates

def _check_lrs(algo, start, delta, tag):
    """Every pair's recorded lrs (last_lrs) against the rule driven by the step's fp64 record KL (last_update_stats), from the
    start lrs {pair: (actor, critic)}; steps the halt skipped have NaN lrs and leave the state.  Returns (borderline steps,
    {pair: (increases, decreases)})."""
    border, moves = 0, {}
    for p in PAIRS:
        lr = [float(np.float32(x)) for x in start[p]]
        rec, st = algo.last_lrs[p], algo.last_update_stats[p]
        assert len(rec) == len(st) > 0, (tag, p)
        assert np.array_equal(rec["epoch"], st["epoch"]) and np.array_equal(rec["minibatch"], st["minibatch"])
        up = down = 0
        for j in range(len(rec)):
            got = [float(rec["actor_lr"][j]), float(rec["critic_lr"][j])]
            if not st["taken"][j]:
                assert all(math.isnan(x) for x in got), (tag, p, j, got)
                continue
            kl = float(st["approx_kl"][j])
            want = [adaptive_lr(x, kl, delta) for x in lr]
            near = any(abs(kl - t) <= 1e-6 * t for t in (2.0 * delta, 0.5 * delta))
            if near:
                border += 1
                assert all(g in (x, w) for g, x, w in zip(got, lr, want)), (tag, p, j, kl, got, lr, want)
            else:
                assert got == want, (tag, p, j, kl, got, want)
            up += got[0] > lr[0]
            down += got[0] < lr[0]
            lr = got
        moves[p] = (up, down)
        oa, oc = dict(algo._pair_optimizers())[p]
        assert [oa.lr, oc.lr] == lr, (tag, p, oa.lr, oc.lr, lr)          # Adam.lr took the final device state
    print("%s: %d steps within 1e-6 of a threshold; (increases, decreases) of the actor lrs per pair %s" % (tag, border, moves))
    return border, moves


def _start(algo):
    return {p: (oa.lr, oc.lr) for p, (oa, oc) in algo._pair_optimizers()}


class _LrSequence:
    """A torch.optim.Adam stand-in for the restatement: the i-th Adam built takes lrs[i][k] as its lr before its k-th step."""

    def __init__(self, lrs):
        self.lrs, self.built, self.adam = list(lrs), 0, torch.optim.Adam

    def __call__(self, params, lr):
        seq = iter(self.lrs[self.built])
        self.built += 1
        opt = self.adam(params, lr=lr)
        step = opt.step

        def stepped():
            opt.param_groups[0]["lr"] = next(seq)
            return step()
        opt.step = stepped
        return opt


@pytest.mark.parametrize("case", ["full", "B3"])
def test_adaptive_update_matches_restatement(mlp_mode, case, monkeypatch):
    """10 full-batch epochs, or 3 epochs x 3 minibatches, at delta = 1e-3: every step's lrs against the rule, the weights against
    the float64 restatement fed the recorded lrs, within tests/test_minibatch_gpu.py's bars for the mode and pair."""
    epochs, B = (10, 1) if case == "full" else (3, 3)
    delta = 1e-3
    algo = _algo(1024, seed=11, n_minibatches=None if case == "full" else B, lr_schedule="adaptive", desired_kl=delta)
    pairs = {0: (algo.actor_net_cross, algo.critic_net_cross), 1: (algo.actor_net_wait, algo.critic_net_wait),
             2: (algo.actor_net_choice, algo.critic_net_choice)}
    sd0 = {w: (_sd64(a), _sd64(c)) for w, (a, c) in pairs.items()}
    start = _start(algo)
    algo.update(epochs=epochs)
    torch.cuda.synchronize()
    _, moves = _check_lrs(algo, start, delta, "mode %d %s" % (mlp_mode, case))
    assert sum(u for u, _ in moves.values()) > 0
    uses_tc = mlp_mode in (0, 2)
    fails = []
    for w, p in enumerate(PAIRS):
        rec = algo.last_lrs[p]
        a, c = pairs[w]
        if a.step == 0:
            continue
        res = {}
        for dtype in (torch.float64, torch.float32):
            monkeypatch.setattr(torch.optim, "Adam", _LrSequence([rec["actor_lr"].tolist(), rec["critic_lr"].tolist()]))
            res[dtype] = _reference_mb_update(algo, w, *sd0[w], epochs, B, dtype=dtype)
            monkeypatch.undo()
        ref, ref32 = res[torch.float64], res[torch.float32]
        assert len(ref["loss_a"]) == len(rec) == a.step
        k32 = 2.0 * ({0: 5.0, 1: 1.0, 2: 25.0}[mlp_mode] if w < 2 else 1.0)
        D = 13 if w < 2 else algo.rollout.shape_env_d
        pk = lambda sd: _pack({k: v.double() for k, v in sd.items()}, D).double().numpy()
        for net, key in ((a, "actor"), (c, "critic")):
            want = pk(ref[key])
            d = np.abs(net.flat.double().cpu().numpy() - want).max() / np.abs(want).max()
            d32 = np.abs(pk(ref32[key]) - want).max() / np.abs(want).max()
            lim = max(2.5e-4 if uses_tc and w < 2 else 1e-4, k32 * d32)
            if mlp_mode == 2 and w < 2 and key == "actor":
                lim = max(lim, 2e-3)
            print("mode %d %s pair %s %s weights: %.3g of the largest (fp32 autograd %.3g, limit %.3g)" % (mlp_mode, case, p, key, d, d32, lim))
            if d > lim:
                fails.append((p, key, d, lim))
    assert not fails, fails


def test_adaptive_with_clipping(mlp_mode):
    """max_grad_norm on top: each step clips its gradient, then takes the adapted lr (tests/test_grad_clip_gpu.py's restatement of
    the clipped step, fed the recorded lr); the lrs follow the rule."""
    G = 0.5
    algo = _algo(1024, seed=5, lr_schedule="adaptive", desired_kl=1e-3, max_grad_norm=G)
    names = {id(a): p for p, a, _ in algo._pair_nets()}
    steps = {p: [] for p in PAIRS}
    sp = algo._step_pair

    def wrap(actor, critic, *a):
        before = [dict(p=n.flat.cpu().numpy(), m=n.m.cpu().numpy(), v=n.v.cpu().numpy(), step=n.step) for n in (actor, critic)]
        sp(actor, critic, *a)
        after = [dict(p=n.flat.cpu().numpy(), m=n.m.cpu().numpy(), v=n.v.cpu().numpy(), g=n.grad.cpu().numpy()) for n in (actor, critic)]
        steps[names[id(actor)]].append((before, after))
    algo._step_pair = wrap
    start = _start(algo)
    algo.update(epochs=3)
    torch.cuda.synchronize()
    _check_lrs(algo, start, 1e-3, "mode %d clip" % mlp_mode)
    clipped = 0
    for p in ("cross", "choice"):
        rec, norms = algo.last_lrs[p], algo.last_grad_norms[p]
        assert len(rec) == len(steps[p]) == len(norms) > 0
        for j, (before, after) in enumerate(steps[p]):
            for y, key in enumerate(("actor_lr", "critic_lr")):
                norm = _close_to_restatement(after[y], before[y], after[y]["g"], float(rec[key][j]), before[y]["step"] + 1, G,
                                             "mode %d %s step %d net %d" % (mlp_mode, p, j, y))
                clipped += norm + 1e-6 > G
    assert clipped > 0


def test_adaptive_with_target_kl(mlp_mode):
    """target_kl on top: the halt test comes first, so a halted step has no lr and leaves the state; Adam.lr ends at the last
    taken step's lr."""
    twin = _algo(2048, target_kl=1e9)
    twin.update(epochs=4)
    torch.cuda.synchronize()
    kl = twin.last_update_stats["cross"]["approx_kl"]
    target = float(kl[1:].max()) / 1.5 * 0.99 if len(kl) > 1 else 1e-9         # halts the cross pair within the update
    algo = _algo(2048, lr_schedule="adaptive", desired_kl=DELTA, target_kl=target)
    start = _start(algo)
    algo.update(epochs=4)
    torch.cuda.synchronize()
    _check_lrs(algo, start, DELTA, "mode %d target_kl" % mlp_mode)
    st = algo.last_update_stats["cross"]
    print("mode %d target_kl: cross steps taken %s" % (mlp_mode, st["taken"].tolist()))
    assert not st["taken"].all()


def test_lr_state_carries_over_and_honours_a_set_lr(mlp_mode):
    algo = _algo(2048, lr_schedule="adaptive", desired_kl=DELTA)
    start = _start(algo)
    algo.update(epochs=3)
    torch.cuda.synchronize()
    _check_lrs(algo, start, DELTA, "mode %d first update" % mlp_mode)
    carried = _start(algo)
    assert carried != start
    algo.update(epochs=3)                                # the same rollout: the second update starts from the first one's lrs
    torch.cuda.synchronize()
    _check_lrs(algo, carried, DELTA, "mode %d second update" % mlp_mode)
    algo.optimizer_actor_cross.lr, algo.optimizer_critic_choice.lr = 2e-3, 5e-5
    set_ = _start(algo)
    algo.update(epochs=3)
    torch.cuda.synchronize()
    _check_lrs(algo, set_, DELTA, "mode %d after setting Adam.lr" % mlp_mode)
    # outside update(): the plain step with Adam.lr, nothing recorded, the lr kept
    before, lr = {p: v.copy() for p, v in algo.last_lrs.items()}, algo.optimizer_actor_cross.lr
    assert algo.train_model_c(algo.actor_net_cross, algo.critic_net_cross, algo.optimizer_actor_cross, algo.optimizer_critic_cross, 0)
    torch.cuda.synchronize()
    assert algo.optimizer_actor_cross.lr == lr and all(before[p].tobytes() == algo.last_lrs[p].tobytes() for p in before)


def test_train_appends_lrs(mlp_mode):
    algo = _algo(512, nb=(1, 1, 1), lr_schedule="adaptive", desired_kl=DELTA)
    algo.train(2, save_traces=False)
    assert len(algo.ep_lrs) == 2 and all(set(it) == set(PAIRS) for it in algo.ep_lrs)
    assert algo.ep_lrs[-1]["choice"]["actor_lr"] == algo.optimizer_actor_choice.lr


# ---------------------------------------------------------------------------------------------------------------------
# 4. two ranks == one rank

def test_two_rank_lrs_equal_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29531", os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "OK" in r.stdout


def _dist_main():
    """Two ranks of N/2 envs against one rank of N envs, "adaptive" at delta = 1e-3, B = 3: the same lrs on every rank, the same
    lrs as one rank except at steps within 1e-6 of a threshold, and the weights within 1e-4 relative."""
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
                                   nb_cars=4, dt=0.3, n_minibatches=3, lr_schedule="adaptive", desired_kl=1e-3)
        algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        algo.update(epochs=3)
        torch.cuda.synchronize()
        return algo
    sharded = run(n, rank * n, True)
    whole = run(N, 0, False)
    for p in PAIRS:
        a, b, st = sharded.last_lrs[p], whole.last_lrs[p], whole.last_update_stats[p]
        t = torch.as_tensor(a.view(np.uint8).copy(), device=dev)
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        assert all(torch.equal(g[0], x) for x in g), "ranks disagree on the lrs"
        near = np.zeros(len(b), dtype=bool)
        for thr in (2e-3, 5e-4):
            near |= np.abs(st["approx_kl"] - thr) <= 1e-6 * thr
        if not near.any():
            assert a.tobytes() == b.tobytes(), p
    worst = 0.0
    for (_, _, ns), (_, _, nw) in zip(sharded._nets(), whole._nets()):
        worst = max(worst, (ns.flat - nw.flat).abs().max().item() / max(nw.flat.abs().max().item(), 1e-12))
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("two-rank lr schedule world=%d: same lrs on every rank and as one rank, max relative weight difference %.3e" % (world, t.item()))
    assert t.item() < 1e-4, t.item()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    _dist_main()
