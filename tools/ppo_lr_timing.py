"""Device time of one full PPO update (Algo_PPO.update, 10 epochs) with each learning-rate schedule, on the scalable 4/3/2 workload
(131 072 envs x 80 steps by default), MLP mode auto (the library's default):

  default      Algo_PPO(): the plain update (mhppo_adam2)
  linear       lr_schedule="linear", lr_anneal_iterations=1000: the same launches with host-set lrs
  adaptive     lr_schedule="adaptive", desired_kl=0.01: the diagnostics' gradient passes and mhppo_adam2_sched
  diagnostics  diagnostics=True alone: what "adaptive" costs beyond its one-CTA Adam launch

Four Algo_PPO instances built alike (same seed, same initial weights).  Each fills its buffers with one rollout; every update then
runs on them (the weights move on, the shapes and routes stay).  The settings alternate within this one process, each repeated
--reps times after a warm-up update.  CUDA events bracket each update, so host gaps inside it and the copies of the lrs count.  The
output gives every sample with the median and the spread, and the library launches of the update.  Then the Adam kernel alone:
mean device time (torch.profiler, CUDA activity) of k_adam2, k_adam2_clip (max_norm inf) and the adaptive k_adam2_clip over --calls
launches each, on the cross pair's nets (4 868 and 4 868 parameters).  The card's name, power limit and max SM clock are read in
the same call.

usage: python tools/ppo_lr_timing.py [--envs N] [--reps R] [--calls K] [--out STEM]     (writes STEM.json and STEM.txt)
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
    modes = [("default", build()), ("linear", build(lr_schedule="linear", lr_anneal_iterations=1000)),
             ("adaptive", build(lr_schedule="adaptive", desired_kl=0.01)), ("diagnostics", build(diagnostics=True))]
    torch.cuda.synchronize()

    def update(algo):
        n0 = mh.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        algo.update()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), mh.launch_count() - n0
    info = {}
    for name, algo in modes:                                     # warm-up of every setting
        _, launches = update(algo)
        info[name] = dict(launches=launches)
    times = {name: [] for name, _ in modes}
    for _ in range(a.reps):
        for name, algo in modes:
            ms, _ = update(algo)
            times[name].append(ms)
    res["update_ms"] = {k: dict(spread(v), **info[k]) for k, v in times.items()}
    for k, v in res["update_ms"].items():
        say("update %-11s median %9.2f ms  min %9.2f  max %9.2f  (%d reps)  launches %d" % (
            k, v["median"], v["min"], v["max"], len(v["samples"]), v["launches"]))
    res["adaptive_lrs_after"] = {p: [oa.lr, oc.lr] for p, (oa, oc) in modes[2][1]._pair_optimizers()}
    say("adaptive: (actor, critic) lrs after the last update", res["adaptive_lrs_after"])

    # the Adam launch alone: the cross pair's nets, gradients of the last update
    plain = modes[0][1]
    act, cri = plain.actor_net_cross, plain.critic_net_cross
    st = torch.cuda.current_stream().cuda_stream
    args = lambda net: (net.flat.data_ptr(), net.grad.data_ptr(), net.m.data_ptr(), net.v.data_ptr(), net.n_param, 1e-12, 1)
    base = args(act) + args(cri) + (0.9, 0.999, 1e-8)
    lr = torch.full((2,), 1e-12, device="cuda")
    kl = torch.full((1,), 0.01 * 1000, device="cuda")        # kl = delta: the lr stays
    lrs = torch.zeros(2, dtype=torch.float64, device="cuda")
    calls = {"adam2": lambda: check(L.mhppo_adam2(*base, st)),
             "adam2_clip_inf": lambda: check(L.mhppo_adam2_clip(*base, math.inf, None, None, 0.0, None, None, st)),
             "adam2_sched": lambda: check(L.mhppo_adam2_sched(*base, math.inf, None, None, 0.0, None, None, lr.data_ptr(), kl.data_ptr(),
                                                              1000.0, 0.01, lrs.data_ptr(), st))}
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
