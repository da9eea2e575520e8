"""Reward normalisation on the GPU (Algo_PPO(normalize_reward=True), mhppo_reward_moments, mhppo_reward_normalize): both entry points
against the float64 restatement of tests/test_reward_norm.py at sizes around every warp, CTA and grid boundary; the update against
the default update fed the normalised rewards (bit for bit, reference mode, GAE, minibatches, diagnostics); the raw learning-curve
traces; one merge per rollout; the coop driver; the launch count; and (two GPUs) two ranks against one.

Bars: batch moments within 1e-12 of the sum of the magnitudes they add, counts exactly, repeated calls bitwise; the merged state
within 1e-12 relative of the restatement fed the kernel's own moments; r~ exactly the restatement from the kernel's own state."""
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

from test_reward_norm import RMS0, batch_moments, merge, running_returns, scale, _rel  # noqa: E402
from test_ppo_diagnostics_gpu import _algo, _state, _same_state, mlp_mode  # noqa: E402,F401

pytestmark = pytest.mark.gpu
EINVAL = -1
GAMMA = 0.99
WS_BYTES = 196608


def _lib():
    import mhppo_b200
    return mhppo_b200.lib()


def _bits(t):
    return t.detach().cpu().contiguous().view(-1).numpy().tobytes()


def _grid_cols():
    """Columns of one full k_reward_moments grid: 8 CTAs of 256 threads per SM."""
    return 8 * torch.cuda.get_device_properties(0).multi_processor_count * 256


def _inputs(T, CN, seed, absent=0.3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    rew = torch.randn(T, CN, generator=g, device="cuda") * 3.0 - 1.0
    rew_d = torch.clamp(torch.randn(CN, generator=g, device="cuda") * 4.0, max=0.0)
    u = torch.rand(CN, generator=g, device="cuda")
    route = torch.where(u < absent, -1, torch.where(u < absent + (1 - absent) / 2, 0, 1)).to(torch.int8)
    return rew.contiguous(), rew_d, route


def _moments(rew, rew_d, route, T, CN, gamma=GAMMA):
    L = _lib()
    out = torch.full((6,), math.nan, dtype=torch.float64, device="cuda")
    ws = torch.zeros(WS_BYTES, dtype=torch.uint8, device="cuda")
    assert L.mhppo_reward_moments(rew.data_ptr(), rew_d.data_ptr(), route.data_ptr(), T, CN, gamma, out.data_ptr(), ws.data_ptr(), None) == 0
    torch.cuda.synchronize()
    return out


def _check_moments(got, rew, rew_d, route, gamma=GAMMA):
    on = route >= 0
    g = running_returns(rew, gamma)[:, on]
    x = rew_d.astype(np.float64)[on]
    want = batch_moments(rew, rew_d, route, gamma)
    assert got[0] == want[0] and got[3] == want[3], (got, want)
    bars = (np.abs(g).sum(), (g * g).sum(), np.abs(x).sum(), (x * x).sum())
    for j, b in zip((1, 2, 4, 5), bars):
        assert abs(got[j] - want[j]) <= 1e-12 * b, (j, got[j], want[j], b)


# ---------------------------------------------------------------------------------------------------------------------
# 1. mhppo_reward_moments

CNS = [1, 31, 32, 33, 255, 256, 257, "grid-1", "grid+1", 4096 * 256 + 257]


@pytest.mark.parametrize("T", [1, 7, 8, 9, 80])
@pytest.mark.parametrize("cn", CNS, ids=str)
def test_reward_moments_match_fp64(cn, T):
    CN = _grid_cols() + (1 if cn == "grid+1" else -1) if isinstance(cn, str) else cn
    rew, rew_d, route = _inputs(T, CN, seed=T * 1000 + CN % 997)
    a = _moments(rew, rew_d, route, T, CN)
    b = _moments(rew, rew_d, route, T, CN)
    assert _bits(a) == _bits(b)
    _check_moments(a.cpu().numpy(), rew.cpu().numpy(), rew_d.cpu().numpy(), route.cpu().numpy())


def test_reward_moments_every_column_absent():
    T, CN = 9, 1000
    rew, rew_d, route = _inputs(T, CN, seed=4, absent=1.0)
    assert (route < 0).all()
    assert (_moments(rew, rew_d, route, T, CN).cpu().numpy() == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# 2. mhppo_reward_normalize

def _normalize(rew, rew_d, T, CN, moments, rms, merge_, clip):
    L = _lib()
    out, out_d = torch.full_like(rew, math.nan), torch.full_like(rew_d, math.nan)
    assert L.mhppo_reward_normalize(rew.data_ptr(), rew_d.data_ptr(), T, CN, moments.data_ptr(), rms.data_ptr(), merge_, clip,
                                    out.data_ptr(), out_d.data_ptr(), None) == 0
    torch.cuda.synchronize()
    return out, out_d


def _check_scaled(out, out_d, rew, rew_d, rms, clip):
    rms = rms.cpu().numpy()
    assert _bits(out) == scale(rew.cpu().numpy(), rms[0][2], clip).tobytes()
    assert _bits(out_d) == scale(rew_d.cpu().numpy(), rms[1][2], clip).tobytes()


@pytest.mark.parametrize("clip", [10.0, 0.3, math.inf])
@pytest.mark.parametrize("T,CN", [(1, 257), (80, 33), (80, 524288)])
def test_reward_normalize_matches_restatement(T, CN, clip):
    rew, rew_d, route = _inputs(T, CN, seed=CN + T)
    rew[0, :5] = torch.tensor([1e3, -1e3, 0.0, -0.0, 3e-39])          # outliers, zeros and a denormal
    mom = _moments(rew, rew_d, route, T, CN)
    start = np.array([[50.0, -4.0, 9.0], [1e-4, 0.0, 1.0]])
    rms = torch.tensor(start, dtype=torch.float64, device="cuda")
    out, out_d = _normalize(rew, rew_d, T, CN, mom, rms, 1, clip)
    want = merge(start, mom.cpu().numpy())
    got = rms.cpu().numpy()
    assert (got[:, 0] == want[:, 0]).all() and (_rel(got[:, 1:], want[:, 1:]) <= 1e-12).all(), (got, want)
    _check_scaled(out, out_d, rew, rew_d, rms, clip)
    if clip < 1:
        assert (out.abs() == float(np.float32(clip))).any() and (out_d.abs() == float(np.float32(clip))).any()
    # merge = 0: the state stays bit for bit, the outputs come from it
    before = _bits(rms)
    out2, out2_d = _normalize(rew, rew_d, T, CN, mom, rms, 0, clip)
    assert _bits(rms) == before and _bits(out2) == _bits(out) and _bits(out2_d) == _bits(out_d)


def test_reward_normalize_empty_batch_keeps_the_state():
    T, CN = 7, 300
    rew, rew_d, route = _inputs(T, CN, seed=8, absent=1.0)
    mom = _moments(rew, rew_d, route, T, CN)
    rms = torch.tensor([[12.5, -3.0, 7.0], [3.0, -1.0, 0.25]], dtype=torch.float64, device="cuda")
    before = _bits(rms)
    out, out_d = _normalize(rew, rew_d, T, CN, mom, rms, 1, 10.0)
    assert _bits(rms) == before
    _check_scaled(out, out_d, rew, rew_d, rms, 10.0)


def test_reward_entry_points_reject_bad_arguments():
    L = _lib()
    T, CN = 4, 64
    rew, rew_d, route = _inputs(T, CN, seed=1)
    mom = torch.zeros(6, dtype=torch.float64, device="cuda")
    rms = torch.tensor(RMS0, dtype=torch.float64, device="cuda")
    ws = torch.zeros(WS_BYTES, dtype=torch.uint8, device="cuda")
    out, out_d = torch.zeros_like(rew), torch.zeros_like(rew_d)
    m = [rew.data_ptr(), rew_d.data_ptr(), route.data_ptr(), T, CN, GAMMA, mom.data_ptr(), ws.data_ptr(), None]
    for i in (0, 1, 2, 6, 7):
        a = list(m); a[i] = None
        assert L.mhppo_reward_moments(*a) == EINVAL, i
    for i, v in ((3, 0), (3, -1), (4, 0), (5, -0.01), (5, 1.01), (5, math.nan)):
        a = list(m); a[i] = v
        assert L.mhppo_reward_moments(*a) == EINVAL, (i, v)
    n = [rew.data_ptr(), rew_d.data_ptr(), T, CN, mom.data_ptr(), rms.data_ptr(), 1, 10.0, out.data_ptr(), out_d.data_ptr(), None]
    for i in (0, 1, 4, 5, 8, 9):
        a = list(n); a[i] = None
        assert L.mhppo_reward_normalize(*a) == EINVAL, i
    for i, v in ((2, 0), (3, 0), (7, 0.0), (7, -1.0), (7, math.nan), (7, -math.inf)):
        a = list(n); a[i] = v
        assert L.mhppo_reward_normalize(*a) == EINVAL, (i, v)
    torch.cuda.synchronize()
    assert _bits(rms) == np.asarray(RMS0, dtype=np.float64).tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the update

SETTINGS = {"full": {}, "gae": dict(gae_lambda=0.95), "B4": dict(n_minibatches=4), "diagnostics": dict(diagnostics=True)}


def _feed_normalised(default, normalised):
    """Let the default Algo_PPO `default` train on `normalised`'s r~ and r~_d: r~ in place of its raw rew buffer, and r~_d in place
    of the rew_d its futur_rewards forms."""
    r, n = default.rollout, normalised.rollout
    r.rew.copy_(n.rew_n)
    plain = r.futur_rewards

    def futur_rewards(rew=None):
        out = plain(rew)
        r.rew_d.copy_(n.rew_dn)
        return out
    r.futur_rewards = futur_rewards


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_update_is_the_default_update_on_normalised_rewards(mlp_mode, setting):
    opts = SETTINGS[setting]
    a = _algo(2048, normalize_reward=True, **opts)
    b = _algo(2048, **opts)
    raw = (_bits(a.rollout.rew), _bits(a.rollout.rl))
    a.update()
    torch.cuda.synchronize()
    r = a.rollout
    assert (_bits(r.rew), _bits(r.rl)) == raw                       # the raw buffers keep their values
    rms = a.reward_rms.cpu().numpy()
    _check_scaled(r.rew_n, r.rew_dn, r.rew, r.rew_d, a.reward_rms, 10.0)
    assert not np.array_equal(r.rew_n.cpu().numpy(), r.rew.cpu().numpy())
    _feed_normalised(b, a)
    b.update()
    torch.cuda.synchronize()
    assert _same_state(_state(a), _state(b)), setting
    assert _bits(a._loss) == _bits(b._loss)
    if setting == "diagnostics":
        assert all(a.last_update_stats[p].tobytes() == b.last_update_stats[p].tobytes() for p in ("cross", "wait", "choice"))
    for k, row in zip(("continuous", "choice"), rms):
        assert a.last_reward_norm[k] == dict(count=row[0], mean=row[1], var=row[2], scale=math.sqrt(row[2] + 1e-8))


def test_learning_curve_traces_stay_raw(mlp_mode):
    a = _algo(1024, normalize_reward=True, clip_reward=math.inf)
    b = _algo(1024)
    a.train(2, save_traces=False)
    b.train(1, save_traces=False)
    torch.cuda.synchronize()
    for k in ("ep_reward_cross", "ep_reward_wait", "ep_reward_choice", "ep_scenario_balance"):
        assert getattr(a, k)[0] == getattr(b, k)[0], k
    assert len(a.ep_reward_norm) == 2 and a.ep_reward_norm[-1] == a.last_reward_norm
    assert a.ep_reward_norm[0]["continuous"]["count"] < a.ep_reward_norm[1]["continuous"]["count"]
    assert b.reward_rms is None and b.ep_reward_norm == [] and b.rollout.rew_n is None


def test_one_merge_per_rollout_and_a_set_state_is_honoured(mlp_mode):
    a = _algo(2048, normalize_reward=True)
    r = a.rollout
    a.update(epochs=1)
    torch.cuda.synchronize()
    mom = a._rn_moments.cpu().numpy()
    _check_moments(mom, r.rew.view(r.T, r.M).cpu().numpy(), r.rew_d.cpu().numpy(), r.route.view(-1).cpu().numpy(), a.gamma)
    first = a.reward_rms.cpu().numpy()
    want = merge(RMS0, mom)
    assert (first[:, 0] == want[:, 0]).all() and (_rel(first[:, 1:], want[:, 1:]) <= 1e-12).all()
    rew_n, rtg = _bits(r.rew_n), _bits(r.rtg)
    a.update(epochs=1)                                   # the same rollout: no second merge, the same r~
    torch.cuda.synchronize()
    assert _bits(a.reward_rms) == first.tobytes() and _bits(r.rew_n) == rew_n and _bits(r.rtg) == rtg
    a.reward_rms[0, 2] = 4.0                             # a state set between updates is honoured
    a.reward_rms[1] = torch.tensor([7.0, -2.0, 0.5], dtype=torch.float64)
    set_ = a.reward_rms.clone()
    a.update(epochs=1)
    torch.cuda.synchronize()
    assert _bits(a.reward_rms) == _bits(set_)
    _check_scaled(r.rew_n, r.rew_dn, r.rew, r.rew_d, set_, 10.0)
    r.iterations_rand(a.actor_net_cross, a.actor_net_wait, a.actor_net_choice)       # a new rollout merges into the set state
    a.update(epochs=1)
    torch.cuda.synchronize()
    want = merge(set_.cpu().numpy(), a._rn_moments.cpu().numpy())
    got = a.reward_rms.cpu().numpy()
    assert (got[:, 0] == want[:, 0]).all() and (_rel(got[:, 1:], want[:, 1:]) <= 1e-12).all()


def test_coop_driver(mlp_mode):
    """The coop (legacy) driver: every car is present, so the batch is every column."""
    import mhppo_b200 as mh
    c, p, l, N = 2, 1, 2, 512
    env = mh.VecCrosswalkEnv("coop", N, nb_car=c, nb_ped=p, nb_lines=l, seed=13, env_id0=2000)
    torch.manual_seed(0)
    a = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=2 + 5 * (c - 1) + 10, num_actions=1, mean=-1.0, std=3.0, nb_cars=c,
                    dt=0.3, normalize_reward=True, clip_reward=5.0)
    r = a.rollout
    r.iterations_rand(a.actor_net_cross, a.actor_net_wait, a.actor_net_choice)
    before = [n.flat.clone() for _, _, n in a._nets()]
    a.update()
    torch.cuda.synchronize()
    assert (r.route >= 0).all()
    rms = a.reward_rms.cpu().numpy()
    assert rms[0][0] == 1e-4 + r.T * r.M and rms[1][0] == 1e-4 + r.M
    mom = batch_moments(r.rew.view(r.T, r.M).cpu().numpy(), r.rew_d.cpu().numpy(), r.route.view(-1).cpu().numpy(), a.gamma)
    want = merge(RMS0, mom)
    assert (_rel(rms[:, 1:], want[:, 1:]) <= 1e-12).all(), (rms, want)
    _check_scaled(r.rew_n, r.rew_dn, r.rew, r.rew_d, a.reward_rms, 5.0)
    assert all(torch.isfinite(n.flat).all() and not torch.equal(n.flat, b) for (_, _, n), b in zip(a._nets(), before)
               if n.step > 0)


def test_update_launches(mlp_mode):
    import mhppo_b200 as mh
    counts = {}
    for name, opts in (("default", {}), ("normalize_reward", dict(normalize_reward=True))):
        a = _algo(2048, **opts)
        for k in ("first", "repeat"):
            n0 = mh.launch_count()
            a.update()
            torch.cuda.synchronize()
            counts[name, k] = mh.launch_count() - n0
    print("launches per update at 4/3/2:", counts)
    assert counts["default", "first"] == counts["default", "repeat"] == 151
    assert counts["normalize_reward", "first"] == 156               # moments (2), merge, scale, reward-to-go from r~
    assert counts["normalize_reward", "repeat"] == 155              # the same rollout: no merge


# ---------------------------------------------------------------------------------------------------------------------
# 4. two ranks == one rank

def test_two_rank_reward_norm_equals_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "OK" in r.stdout


def _dist_main():
    """Two ranks of N/2 envs against one rank of N envs, two rollouts with one update each: the same reward_rms on every rank,
    within 1e-12 relative of one rank's, and the weights within 1e-4 relative."""
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
                                   nb_cars=4, dt=0.3, normalize_reward=True)
        for _ in range(2):
            algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
            algo.update(epochs=3)
        torch.cuda.synchronize()
        return algo
    sharded = run(n, rank * n, True)
    whole = run(N, 0, False)
    g = [torch.zeros_like(sharded.reward_rms) for _ in range(world)]
    dist.all_gather(g, sharded.reward_rms)
    assert all(_bits(g[0]) == _bits(x) for x in g), "ranks disagree on reward_rms"
    a, b = sharded.reward_rms.cpu().numpy(), whole.reward_rms.cpu().numpy()
    assert (a[:, 0] == b[:, 0]).all() and (_rel(a[:, 1:], b[:, 1:]) <= 1e-12).all(), (a, b)
    worst = 0.0
    for (_, _, ns), (_, _, nw) in zip(sharded._nets(), whole._nets()):
        worst = max(worst, (ns.flat - nw.flat).abs().max().item() / max(nw.flat.abs().max().item(), 1e-12))
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("two-rank reward normalisation world=%d: same reward_rms on every rank, as one rank within 1e-12, max relative weight "
              "difference %.3e" % (world, t.item()))
    assert t.item() < 1e-4, t.item()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    _dist_main()
