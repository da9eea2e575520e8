"""Device time of one full PPO update (Algo_PPO.update, 10 epochs) with and without the update diagnostics, on the scalable 4/3/2
workload (131 072 envs x 80 steps by default), MLP mode auto (the library's default):

  default      Algo_PPO(diagnostics=False, target_kl=None): the plain update, on an instance of its own
  diag         diagnostics=True
  kl_never     diagnostics=True, target_kl=1e9 (the halting Adam step runs; 1.5e9 is far above any step's KL)
  kl_small     diagnostics=True, target_kl=1e-3, a small value meant to fire: the output reports the steps each pair took

Two Algo_PPO instances built alike (same seed, same initial weights): one plain, one with diagnostics, whose target_kl is switched
between updates.  Each fills its buffers with one rollout; every update then runs on them (the weights move on, the shapes and
routes stay).  The settings alternate within this one process, each repeated --reps times after a warm-up update.  CUDA events
bracket each update, so host gaps inside it and the record copy count.  The output gives every sample with the median and the
spread, the Adam steps each pair took and the library launches of the update.  The card's name, power limit and max SM clock
are read in the same call.

usage: python tools/ppo_diag_timing.py [--envs N] [--reps R] [--out STEM]     (writes STEM.json and STEM.txt)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "samples": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import mhppo_b200 as mh
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
    plain, diag = build(), build(diagnostics=True)
    torch.cuda.synchronize()

    def update(algo, target_kl):
        if algo is diag:
            algo.target_kl = target_kl
            algo._check_options()
        actors = [x for _, x, _ in algo._pair_nets()]
        s0, n0 = [x.step for x in actors], mh.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        algo.update()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), [x.step - s for x, s in zip(actors, s0)], mh.launch_count() - n0
    modes = [("default", plain, None), ("diag", diag, None), ("kl_never", diag, 1e9), ("kl_small", diag, 1e-3)]
    info = {}
    for name, algo, t in modes:                                  # warm-up of every setting
        _, steps, launches = update(algo, t)
        info[name] = dict(launches=launches, target_kl=t)
    times = {name: [] for name, _, _ in modes}
    taken = {name: [] for name, _, _ in modes}
    for _ in range(a.reps):
        for name, algo, t in modes:
            ms, steps, _ = update(algo, t)
            times[name].append(ms)
            taken[name].append(steps)
    res["update_ms"] = {k: dict(spread(v), adam_steps_taken_cross_wait_choice=taken[k], **info[k]) for k, v in times.items()}
    for k, v in res["update_ms"].items():
        say("update %-8s median %9.2f ms  min %9.2f  max %9.2f  (%d reps)  launches %d  Adam steps taken (cross, wait, choice) per rep %s" % (
            k, v["median"], v["min"], v["max"], len(v["samples"]), v["launches"], v["adam_steps_taken_cross_wait_choice"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)) or ".", exist_ok=True)
        with open(a.out + ".json", "w") as f:
            json.dump(res, f, indent=1)
        with open(a.out + ".txt", "w") as f:
            f.write("\n".join(lines) + "\n")
    assert L.mhppo_tc_failures() == 0


if __name__ == "__main__":
    main()
