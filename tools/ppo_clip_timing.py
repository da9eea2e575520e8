"""Device time of one full PPO update (Algo_PPO.update, 10 epochs) with and without per-net gradient-norm clipping, on the
scalable 4/3/2 workload (131 072 envs x 80 steps by default), MLP mode auto (the library's default):

  default      Algo_PPO(max_grad_norm=None): the plain update (mhppo_adam2), on an instance of its own
  clip_inf     max_grad_norm=inf: mhppo_adam2_clip with the norms recorded, never clipping
  clip_0.5     max_grad_norm=0.5 (SB3's default): the same launch, clipping whenever a net's norm exceeds 0.5

Two Algo_PPO instances built alike (same seed, same initial weights): one plain, one whose max_grad_norm is switched between
updates.  Each fills its buffers with one rollout; every update then runs on them (the weights move on, the shapes and routes
stay).  The settings alternate within this one process, each repeated --reps times after a warm-up update.  CUDA events bracket
each update, so host gaps inside it and the copy of the norms count.  The output gives every sample with the median and the
spread, the library launches of the update and the fraction of nets whose step was clipped.  Then, after the timed updates, the
Adam kernel alone: mean device time (torch.profiler, CUDA activity) of k_adam2 and k_adam2_clip over --calls launches each, on the
cross pair's nets (4 868 and 4 868 parameters).  The card's name, power limit and max SM clock are read in the same call.

usage: python tools/ppo_clip_timing.py [--envs N] [--reps R] [--calls K] [--out STEM]     (writes STEM.json and STEM.txt)
"""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from ppo_diag_timing import card, spread  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import mhppo_b200 as mh
    from mhppo_b200._lib import check
    L = mh.lib()
    lines = []

    def say(*args):
        line = " ".join(str(x) for x in args)
        print(line)
        lines.append(line)
    res = {"card": card(), "workload": "coop_scalable nb_car 4 nb_ped 3 nb_lines 2, %d envs x 80 steps, reference mode, MLP mode auto" % a.envs}
    say("card:", res["card"])

    def build(**opts):
        env = mh.VecCrosswalkEnv("coop_scalable", a.envs, nb_car=4, nb_ped=3, nb_lines=2, seed=1, env_id0=0)
        torch.manual_seed(0)
        algo = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=30, num_actions=1, mean=-1.0, std=3.0, nb_cars=4, dt=0.3,
                           **opts)
        algo.rollout.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        return algo
    plain, clip = build(), build(max_grad_norm=math.inf)
    torch.cuda.synchronize()

    def update(algo, g):
        if algo is clip:
            algo.max_grad_norm = g
            algo._check_options()
        n0 = mh.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        algo.update()
        e1.record()
        torch.cuda.synchronize()
        clipped = None
        if algo is clip:
            norms = np.concatenate([np.stack([v["actor_grad_norm"], v["critic_grad_norm"]]).ravel() for v in algo.last_grad_norms.values()])
            clipped = float(np.mean(g / (norms + 1e-6) < 1.0))
        return e0.elapsed_time(e1), mh.launch_count() - n0, clipped
    modes = [("default", plain, None), ("clip_inf", clip, math.inf), ("clip_0.5", clip, 0.5)]
    info = {}
    for name, algo, g in modes:                                  # warm-up of every setting
        _, launches, _ = update(algo, g)
        info[name] = dict(launches=launches, max_grad_norm=str(g))
    times = {name: [] for name, _, _ in modes}
    frac = {name: [] for name, _, _ in modes}
    for _ in range(a.reps):
        for name, algo, g in modes:
            ms, _, c = update(algo, g)
            times[name].append(ms)
            frac[name].append(c)
    res["update_ms"] = {k: dict(spread(v), fraction_of_net_steps_clipped=frac[k], **info[k]) for k, v in times.items()}
    for k, v in res["update_ms"].items():
        say("update %-8s median %9.2f ms  min %9.2f  max %9.2f  (%d reps)  launches %d  fraction of net steps clipped per rep %s" % (
            k, v["median"], v["min"], v["max"], len(v["samples"]), v["launches"], v["fraction_of_net_steps_clipped"]))

    # the Adam launch alone: the cross pair's nets, gradients of the last update
    act, cri = plain.actor_net_cross, plain.critic_net_cross
    st = torch.cuda.current_stream().cuda_stream
    args = lambda net: (net.flat.data_ptr(), net.grad.data_ptr(), net.m.data_ptr(), net.v.data_ptr(), net.n_param, 1e-12, 1)
    base = args(act) + args(cri) + (0.9, 0.999, 1e-8)
    norms = torch.zeros(2, dtype=torch.float64, device="cuda")
    calls = {"adam2": lambda: check(L.mhppo_adam2(*base, st)),
             "adam2_clip_inf": lambda: check(L.mhppo_adam2_clip(*base, math.inf, norms.data_ptr(), None, 0.0, None, None, st)),
             "adam2_clip_0.5": lambda: check(L.mhppo_adam2_clip(*base, 0.5, norms.data_ptr(), None, 0.0, None, None, st))}
    kt = {}
    for k, f in calls.items():
        for _ in range(10):                                      # warm-up
            f()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(a.calls):
                f()
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "k_adam2" in e.key]
        assert len(ev) == 1 and ev[0].count == a.calls, [(e.key, e.count) for e in ev]
        kt[k] = dict(kernel=ev[0].key, mean_us=ev[0].self_device_time_total / ev[0].count, calls=a.calls, n_params=[act.n_param, cri.n_param])
    res["adam_kernel_us"] = kt
    for k, v in kt.items():
        say("kernel %-15s mean device time %7.3f us over %d calls (torch.profiler; nets of %d / %d parameters): %s" % (
            k, v["mean_us"], v["calls"], act.n_param, cri.n_param, v["kernel"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)) or ".", exist_ok=True)
        with open(a.out + ".json", "w") as f:
            json.dump(res, f, indent=1)
        with open(a.out + ".txt", "w") as f:
            f.write("\n".join(lines) + "\n")
    assert L.mhppo_tc_failures() == 0


if __name__ == "__main__":
    main()
