"""Device time of one full PPO update (Algo_PPO.update: 10 epochs of the cross and wait pairs, then 10 of the choice pair) in
reference mode, GAE mode (gae_lambda 0.95) and GAE + entropy bonus (entropy_coef 0.01), and of one mhppo_gae call alone, on
the scalable 4/3/2 workload (131 072 envs x 80 steps by default).

One rollout fills the buffers; every update then runs on them (the weights move on, the shapes and routes stay).  The three
modes alternate within this one process, each repeated --reps times after a warm-up update, and the output gives every
sample with the median and the spread.  CUDA events bracket each update, so host gaps inside it count.  mhppo_gae is timed
over 20 back-to-back calls; its inputs (rewards, V_old, route) and output exceed the 126 MB L2, so they stream from HBM.
Its algorithmic traffic is counted from the routes: 4 B reward + 4 B V_old + 4 B return per sample of a present car, 4 B
(the zero return) per sample of an absent car, and 1 B route per column.  The bound divides that by 7.7 TB/s, the HBM3e
bandwidth of one B200 in NVIDIA's HGX B200 data sheet (not a measured figure).

usage: python tools/ppo_gae_timing.py [--envs N] [--reps R] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12
MODES = [("reference", None, 0.0), ("gae_0.95", 0.95, 0.0), ("gae_0.95+entropy_0.01", 0.95, 0.01)]


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
    from mhppo_b200._lib import check
    res = {"card": card(), "workload": "coop_scalable nb_car 4 nb_ped 3 nb_lines 2, %d envs x 80 steps" % a.envs}
    print("card:", res["card"])
    env = mh.VecCrosswalkEnv("coop_scalable", a.envs, nb_car=4, nb_ped=3, nb_lines=2, seed=1, env_id0=0)
    torch.manual_seed(0)
    algo = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=30, num_actions=1, mean=-1.0, std=3.0, nb_cars=4, dt=0.3)
    r = algo.rollout
    r.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
    torch.cuda.synchronize()

    def update(lam, c):
        algo.gae_lambda, algo.entropy_coef = lam, c
        algo._check_options()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        algo.update()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    for _, lam, c in MODES:                                   # warm-up: modules, shared-memory attributes, GAE buffers
        update(lam, c)
    times = {name: [] for name, _, _ in MODES}
    for _ in range(a.reps):
        for name, lam, c in MODES:
            times[name].append(update(lam, c))
    res["update_ms"] = {k: spread(v) for k, v in times.items()}

    # mhppo_gae alone (k_gae + the 6-value k_reduce_gae), V_old as the last GAE update left it
    L = mh.lib()
    st = torch.zeros(6, dtype=torch.float64, device="cuda")
    ws = algo._ws

    def gae_call():
        check(L.mhppo_gae(r.rew.data_ptr(), r.V.data_ptr(), r.route.data_ptr(), r.T, r.M, 0.99, 0.95, r.ret.data_ptr(), st.data_ptr(),
                          ws.data_ptr(), None))
    gae_call()
    n_calls, gae_ms = 20, []
    for _ in range(max(a.reps, 5)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_calls):
            gae_call()
        e1.record()
        torch.cuda.synchronize()
        gae_ms.append(e0.elapsed_time(e1) / n_calls)
    present = int((r.route >= 0).sum().item())
    nbytes = 12 * r.T * present + 4 * r.T * (r.M - present) + r.M
    g = spread(gae_ms)
    res["mhppo_gae"] = dict(ms=g, columns=r.M, present_columns=present, steps=r.T, algorithmic_bytes=nbytes,
                            hbm_bound_ms=nbytes / HBM_BYTES_PER_S * 1e3, bandwidth_figure="7.7 TB/s (HGX B200 data sheet, per GPU)",
                            achieved_TBps=nbytes / (g["median"] * 1e-3) / 1e12,
                            share_of_bound=(nbytes / HBM_BYTES_PER_S * 1e3) / g["median"])
    for k, v in res["update_ms"].items():
        print("update %-24s median %8.2f ms  min %8.2f  max %8.2f  (%d reps)" % (k, v["median"], v["min"], v["max"], len(v["samples"])))
    m = res["mhppo_gae"]
    print("mhppo_gae: median %.4f ms (min %.4f, max %.4f); %d of %d columns present; %.1f MB algorithmic; bound %.4f ms at 7.7 TB/s; "
          "achieved %.2f TB/s = %.0f %% of the bound" % (g["median"], g["min"], g["max"], present, r.M, nbytes / 1e6, m["hbm_bound_ms"],
                                                        m["achieved_TBps"], 100 * m["share_of_bound"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    assert L.mhppo_tc_failures() == 0


if __name__ == "__main__":
    main()
