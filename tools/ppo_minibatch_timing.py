"""Device time of one full PPO update (Algo_PPO.update, 10 epochs) without minibatches (n_minibatches=None) and with B = 1, 4, 16
and 64 minibatches per epoch, and of one mhppo_minibatch_plan call alone, on the scalable 4/3/2 workload (131 072 envs x 80 steps
by default), reference mode.

One rollout fills the buffers; every update then runs on them (the weights move on, the shapes and routes stay).  The modes
alternate within this one process, each repeated --reps times after a warm-up update; the output gives every sample with the
median and the spread, the Adam steps each update took and the library launches it issued.  CUDA events bracket each update, so
host gaps inside it count.

mhppo_minibatch_plan is timed over 20 back-to-back calls at the workload's size (10 epochs, 524 288 columns: its 63 MB of lists
fit the 126 MB L2) and on a synthetic route of --plan-envs envs x 4 cars (default 1 048 576: 503 MB of lists, larger than the
L2, so the outputs stream to HBM).

usage: python tools/ppo_minibatch_timing.py [--envs N] [--reps R] [--plan-envs N] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MODES = [("none", None), ("B1", 1), ("B4", 4), ("B16", 16), ("B64", 64)]


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


def time_plan(L, check, cfg, route, exist, act_d, E, B, n_calls=20, reps=5):
    import torch
    M = route.numel()
    lists = torch.empty(E * 3 * M, dtype=torch.int32, device="cuda")
    off = torch.empty(E * 3 * (B + 1), dtype=torch.int64, device="cuda")
    cnt = torch.empty(E * 5 * B, dtype=torch.int64, device="cuda")
    ws = torch.empty(1280 * E * B, dtype=torch.uint8, device="cuda")

    def call():
        check(L.mhppo_minibatch_plan(C.byref(cfg), route.data_ptr(), exist.data_ptr(), act_d.data_ptr(), 3, E, B, lists.data_ptr(),
                                     off.data_ptr(), cnt.data_ptr(), ws.data_ptr(), None))
    call()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_calls):
            call()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / n_calls)
    return dict(ms=spread(out), columns=M, epochs=E, buckets=B, list_bytes=4 * 3 * E * M)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--plan-envs", type=int, default=1048576)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import mhppo_b200 as mh
    from mhppo_b200._lib import RolloutCfg, check
    L = mh.lib()
    res = {"card": card(), "workload": "coop_scalable nb_car 4 nb_ped 3 nb_lines 2, %d envs x 80 steps, reference mode" % a.envs}
    print("card:", res["card"])
    env = mh.VecCrosswalkEnv("coop_scalable", a.envs, nb_car=4, nb_ped=3, nb_lines=2, seed=1, env_id0=0)
    torch.manual_seed(0)
    algo = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=30, num_actions=1, mean=-1.0, std=3.0, nb_cars=4, dt=0.3)
    r = algo.rollout
    r.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
    torch.cuda.synchronize()
    nets = [net for _, _, net in algo._nets()]

    def update(B):
        algo.n_minibatches = B
        algo._check_options()
        s0, n0 = [n.step for n in nets], mh.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        algo.update()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), [n.step - s for n, s in zip(nets, s0)][:3], mh.launch_count() - n0
    info = {}
    for name, B in MODES:                                     # warm-up: modules, plan buffers
        _, steps, launches = update(B)
        info[name] = dict(adam_steps_cross_wait_choice=steps, launches=launches)
    times = {name: [] for name, _ in MODES}
    for _ in range(a.reps):
        for name, B in MODES:
            times[name].append(update(B)[0])
    res["update_ms"] = {k: dict(spread(v), **info[k]) for k, v in times.items()}

    res["plan_workload"] = {}
    for _, B in MODES[1:]:
        res["plan_workload"]["B%d" % B] = time_plan(L, check, r._cfg, r.route, r.exist, r.act_d, 10, B)
    big = a.plan_envs
    g = torch.Generator(device="cuda").manual_seed(5)
    route = (torch.randint(0, 4, (4, big), device="cuda", generator=g) - 1).clamp(max=1).to(torch.int8)
    exist = (route >= 0).to(torch.int8)
    act_d = torch.randint(0, 2, (4 * big,), device="cuda", generator=g).float()
    cfg = RolloutCfg(nb_ped=3, nb_lines=2, T=80, legacy_nb_car=0, n_envs=big, seed=1, env_id0=0)
    res["plan_large"] = {"B%d" % B: time_plan(L, check, cfg, route, exist, act_d, 10, B) for B in (16, 1024)}

    for k, v in res["update_ms"].items():
        print("update %-5s median %9.2f ms  min %9.2f  max %9.2f  (%d reps)  Adam steps %s  launches %d" % (
            k, v["median"], v["min"], v["max"], len(v["samples"]), v["adam_steps_cross_wait_choice"], v["launches"]))
    for grp in ("plan_workload", "plan_large"):
        for k, v in res[grp].items():
            print("mhppo_minibatch_plan %-13s %-5s %8d columns x 10 epochs (%6.1f MB of lists): median %.4f ms (min %.4f, max %.4f)" % (
                grp, k, v["columns"], v["list_bytes"] / 1e6, v["ms"]["median"], v["ms"]["min"], v["ms"]["max"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    assert L.mhppo_tc_failures() == 0


if __name__ == "__main__":
    main()
