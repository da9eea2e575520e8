"""Device time of one full PPO update (Algo_PPO.update, 10 epochs) with and without reward normalisation, on the scalable 4/3/2
workload (131 072 envs x 80 steps by default), MLP mode auto (the library's default):

  default           Algo_PPO(): the plain update
  normalize_reward  normalize_reward=True: + mhppo_reward_moments, mhppo_reward_normalize and the reward-to-go from r~

Two Algo_PPO instances built alike (same seed, same initial weights).  Each fills its buffers with one rollout; every update then
runs on them (the weights move on, the shapes and routes stay), so after the warm-up each normalised update is a repeat on the same
rollout: it computes and all-reduces the batch moments but does not merge them (no k_reward_merge launch).  The settings alternate
within this one process, each repeated --reps times after a warm-up update.  CUDA events bracket each update, so host gaps inside it
and the copy of reward_rms count.  The output gives every sample with the median and the spread, and the library launches of the
warm-up (first) update and of a repeat.

Then the two entry points alone, on the normalised instance's buffers (rew [S] = 167.8 MB at the default size, more than the 126 MB
L2): --calls back-to-back calls each between CUDA events, mean time per call, and the bytes each call must move over that time
against 7.7 TB/s:
  mhppo_reward_moments             reads rew [S] fp32, rew_d [M] fp32, route [M] int8
  mhppo_reward_normalize, merge=1  reads rew, rew_d; writes rew_n [S], rew_dn [M] (the one-thread merge launch first)
The card's name, power limit and max SM clock are read in the same call.

usage: python tools/ppo_reward_norm_timing.py [--envs N] [--reps R] [--calls K] [--out STEM]     (writes STEM.json and STEM.txt)
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from ppo_diag_timing import card, spread  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
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
    modes = [("default", build()), ("normalize_reward", build(normalize_reward=True))]
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
    for name, algo in modes:                                     # warm-up of every setting (the normalised one merges here)
        _, launches = update(algo)
        info[name] = dict(launches_first=launches)
    times = {name: [] for name, _ in modes}
    for _ in range(a.reps):
        for name, algo in modes:
            ms, launches = update(algo)
            times[name].append(ms)
            info[name]["launches_repeat"] = launches
    res["update_ms"] = {k: dict(spread(v), **info[k]) for k, v in times.items()}
    for k, v in res["update_ms"].items():
        say("update %-16s median %9.2f ms  min %9.2f  max %9.2f  (%d reps)  launches: first update %d, repeat %d" % (
            k, v["median"], v["min"], v["max"], len(v["samples"]), v["launches_first"], v["launches_repeat"]))
    norm = modes[1][1]
    res["reward_norm_after"] = norm.last_reward_norm
    say("reward_rms after the updates:", norm.last_reward_norm)

    # the two entry points alone, on the normalised instance's buffers
    r = norm.rollout
    st = torch.cuda.current_stream().cuda_stream
    mom, rms = torch.zeros(6, dtype=torch.float64, device="cuda"), norm.reward_rms.clone()
    S, M = r.S, r.M
    calls = {"reward_moments": (lambda: check(L.mhppo_reward_moments(r.rew.data_ptr(), r.rew_d.data_ptr(), r.route.data_ptr(), r.T, M,
                                                                     0.99, mom.data_ptr(), norm._ws.data_ptr(), st)),
                                4 * S + 4 * M + M),
             "reward_normalize_merge": (lambda: check(L.mhppo_reward_normalize(r.rew.data_ptr(), r.rew_d.data_ptr(), r.T, M, mom.data_ptr(),
                                                                               rms.data_ptr(), 1, 10.0, r.rew_n.data_ptr(),
                                                                               r.rew_dn.data_ptr(), st)),
                                        2 * (4 * S + 4 * M))}
    kt = {}
    for k, (f, nbytes) in calls.items():
        for _ in range(3):                                       # warm-up
            f()
        torch.cuda.synchronize()
        n0 = mh.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.calls):
            f()
        e1.record()
        torch.cuda.synchronize()
        us = 1e3 * e0.elapsed_time(e1) / a.calls
        kt[k] = dict(mean_us=us, calls=a.calls, launches_per_call=(mh.launch_count() - n0) // a.calls, bytes=nbytes,
                     achieved_TBps=nbytes / (us * 1e-6) / 1e12, fraction_of_7_7_TBps=nbytes / (us * 1e-6) / HBM_BYTES_PER_S)
    res["entry_points"] = kt
    for k, v in kt.items():
        say("%-23s %8.2f us per call over %d back-to-back calls (CUDA events, %d launches per call); %.1f MB -> %.2f TB/s = %.0f%% of 7.7 TB/s"
            % (k, v["mean_us"], v["calls"], v["launches_per_call"], v["bytes"] / 1e6, v["achieved_TBps"], 100 * v["fraction_of_7_7_TBps"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)) or ".", exist_ok=True)
        with open(a.out + ".json", "w") as f:
            json.dump(res, f, indent=1)
        with open(a.out + ".txt", "w") as f:
            f.write("\n".join(lines) + "\n")
    assert L.mhppo_tc_failures() == 0


if __name__ == "__main__":
    main()
