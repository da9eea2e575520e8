#!/usr/bin/env python
"""bench.py -- headline benchmark of the MH-PPO hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Metric (BASELINE.json): agent-steps/sec of env.step.  A "step" is one env.step over the whole batch
of synthetic envs held by a GPU.  Default workload = the configuration the north-star target is
quoted on: Env_hybrid_multi_coop_scalable, nb_car=4 / nb_ped=3 / nb_lines=2, 262144 envs per GPU
(BASELINE.json configs[3]); envs shard across ranks with no data-path collective ("weak" scaling).

`value`  : device-timed (CUDA events on the launching stream, one pair per step, max over ranks),
           inputs resident in HBM, L2 flushed (untimed 256 MiB memset) between timed steps.
`e2e`    : the same metric through the reference-facing call with HOST buffers
           (mhppo_env_step_host: numpy-in/numpy-out convention of env.step): H2D of the actions and
           D2H of obs/rewards/reward_light/done inside the timed region.
`roofline`: algorithmic bytes per env-step (SURVEY.md 8d: B = 2*(32C+64P+16) + 8*C_act + 8*C +
           4*obs_floats + 4) x envs / mean kernel time, against MEASURED_PEAKS.json hbm_gbs.
`cpu_baseline`: the C oracle port (oracle/, the only CPU code; test infrastructure) timed on this
           box's host cores on a bounded sample of the same workload.
--impl reference: the reference's own CPU path.  The reference is pure Python and cannot travel to
the GPU box; the arm times the pinned C restatement (oracle port) with all host threads.
--dump-outputs DIR: after the timed region, what the last timed env.step returned (env_step_*.npy) and, when the PPO
section runs, what its last timed iteration left to the caller: rollout buffers and updated networks (ppo_*.npy); a
fixed, seeded sample of the envs (DUMP_ENVS), float32 / float64, at most 64 MB in all.  The inputs are seeded, so two
builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (it may be read-only)

WORKLOADS = {
    # name: (variant, nb_car, nb_ped, nb_lines, envs per GPU)
    "scalable_432": ("coop_scalable", 4, 3, 2, 262144),      # BASELINE configs[3] (north-star target)
    "coop_212": ("coop", 2, 1, 2, 4096),                     # configs[1]
    "4cars_222": ("coop_4cars", 2, 2, 2, 65536),             # configs[2]
    "stop_121": ("stop", 1, 2, 1, 4096),                     # configs[0] shape, batched
}


def algorithmic_bytes(variant, nb_car, nb_ped, nb_lines):
    """SURVEY.md 8(d) per-env-step figure."""
    if variant == "coop_scalable":
        C, C_act, carw, envw = 2 * nb_lines, 2 * nb_lines, 7, 4
    elif "4cars" in variant:
        C, C_act, carw, envw = 2 * nb_car, (2 * nb_car if variant.endswith("2") else nb_car), 6, 3
    else:
        C, C_act, carw, envw = nb_car, nb_car, 6, 3
    obs = carw * C + envw + 9 * nb_ped
    S = 32 * C + 64 * nb_ped + 16
    return 2 * S + 8 * C_act + 8 * C + 4 * obs + 4, C, obs


TRAFFIC_FILES = ("round2_env_step_ncu_metrics.json", "round1_env_step_ncu_metrics.json")      # newest capture first


def recorded_traffic(n_envs):
    """dram__bytes_read.sum + dram__bytes_write.sum of k_env_step from the committed ncu --set full capture."""
    for name in TRAFFIC_FILES:
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            if int(d["n_envs"]) == int(n_envs):
                return d["traffic_bytes_per_launch"], "profiles/%s (ncu --set full, bytes per launch)" % name
        except Exception:
            continue
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy burst)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi SM clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()

    def run(self):
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            self._stop_ev.wait(0.2)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


EPISODE = 80   # every episode of every env class lasts exactly 80 steps (SURVEY.md section 6)


def synthetic_actions_np(n_envs, A, seed=0):
    """SURVEY.md 8(d): acc ~ U(-4, 2) fresh every step (a pool of 4 draws, cycled), light in {-1, +1} drawn once per
    episode and held for its 80 steps (two light draws, alternating from one episode to the next)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lights = [rng.choice([-1.0, 1.0], (n_envs, A // 2)) for _ in range(2)]
    acts = []
    for e in range(2):
        row = []
        for _ in range(4):
            a = np.empty((n_envs, A))
            a[:, :A // 2] = rng.uniform(-4, 2, (n_envs, A // 2))
            a[:, A // 2:] = lights[e]
            row.append(a)
        acts.append(row)
    return acts


DUMP_ENVS = {"env_step": 32768, "ppo": 1024}   # envs sampled into --dump-outputs (16.8 + 25.5 MB at the default sizes)
DUMP_LIMIT = 64 << 20
_dumped_bytes = 0


def dump_envs(n_envs, k):
    """Ascending indices of a fixed, seeded sample of k of the n_envs envs (all of them when n_envs <= k)."""
    import numpy as np
    return np.arange(n_envs) if n_envs <= k else np.sort(np.random.default_rng(0).choice(n_envs, k, replace=False))


def write_dump(out_dir, arrays):
    """--dump-outputs: each tensor of `arrays` to out_dir/<name>.npy; float64 stays float64, everything else is float32."""
    import numpy as np
    global _dumped_bytes
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a if a.dtype == np.float64 else a.astype(np.float32)
        _dumped_bytes += a.nbytes
        if _dumped_bytes > DUMP_LIMIT:
            raise RuntimeError("--dump-outputs would exceed %d MB (at %s.npy)" % (DUMP_LIMIT >> 20, name))
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_port_run(variant, nb_car, nb_ped, nb_lines, n_envs, warmup, steps, threads=0, min_seconds=5.0, max_rounds=64):
    """The CPU leg of both arms: the C oracle port on the host cores over the WHOLE n_envs batch.  One round = reset,
    `warmup` untimed steps, `steps` timed steps (the same window of the episode the GPU arm times); rounds are repeated
    until `min_seconds` of timed work.  Returns (env-steps/s, timed seconds, active agents per env, rounds)."""
    import numpy as np
    from oracle import oracle as O
    env = O.OracleVecEnv(variant, n_envs, nb_car, nb_ped, nb_lines, seed=1234, n_threads=threads, store_f32=False)
    A = env.n_action
    acts = synthetic_actions_np(n_envs, A)
    obs = np.empty((n_envs, env.n_obs), np.float32)
    rew = np.empty((n_envs, env.n_lead)); rl = np.empty((n_envs, env.n_lead)); done = np.empty(n_envs, np.uint8)
    timed, rounds, active = 0.0, 0, []
    while rounds < max_rounds and (rounds == 0 or timed < min_seconds):
        env.reset()
        for t in range(warmup):
            env.step_into(acts[(t // EPISODE) % 2][t % 4], obs, rew, rl, done)
        t0 = time.perf_counter()
        for t in range(warmup, warmup + steps):
            env.step_into(acts[(t // EPISODE) % 2][t % 4], obs, rew, rl, done)
        timed += time.perf_counter() - t0
        rounds += 1
        s = env.get_state()
        active.append(float((s["env_i"][:, 1] + s["env_i"][:, 2]).mean()))
    return n_envs * steps * rounds / timed, timed, sum(active) / len(active), rounds


def cpu_ppo_rate(n_envs=256, wl=("coop_scalable", 4, 3, 2)):
    """PPO samples/s of the CPU restatement of the PPO pipeline (oracle/ppo_oracle.py: vectorised numpy feature builders,
    torch CPU networks / autograd / Adam on all host threads, C env port): one iteration = one 80-step episode per env,
    reward-to-go, 10 x (cross, wait) + 10 x choice epochs (Algo_PPO.train, PY:854-917)."""
    import numpy as np
    import torch
    from oracle import oracle as O, ppo_oracle as PO
    torch.manual_seed(0)
    variant, nb_car, P, L = wl
    seed = 1234
    legacy = 0 if variant == "coop_scalable" else nb_car
    D = 2 + (5 * (nb_car - 1) if legacy else 6 * (2 * L - 1)) + 8 + 2
    actors = [PO.Net(13, 1, 1), PO.Net(13, 1, 1), PO.Net(D, 2, 2)]
    critics = [PO.Net(13, 1, 0), PO.Net(13, 1, 0), PO.Net(D, 1, 0)]
    opt_a = [torch.optim.Adam(n.parameters(), lr=3e-4) for n in actors]
    opt_c = [torch.optim.Adam(n.parameters(), lr=1e-3) for n in critics]
    env = O.OracleVecEnv(variant, n_envs, nb_car, P, L, seed=seed, store_f32=False)
    t0 = time.perf_counter()
    sds = [{k: v.detach().clone() for k, v in n.state_dict().items()} for n in actors]
    b = PO.rollout_episode(env, *sds, seed, np.arange(n_envs), P, L, legacy_nb_car=legacy)
    rtg = PO.reward_to_go(b["rew"])
    t_roll = time.perf_counter() - t0
    n_samples = 0
    for k in (0, 1):                                                        # cross, wait (PY:868-877)
        m = b["route"] == k                                                 # [C, N]
        if not m.any():
            continue
        st, ac, lp, rt = b["obs_c"][:, m], b["act"][:, m], b["logp"][:, m], rtg[:, m]
        st, ac, lp, rt = st.reshape(-1, 13), ac.reshape(-1), lp.reshape(-1), rt.reshape(-1)
        n_samples += st.shape[0]
        for _ in range(10):
            PO.train_step_c(actors[k], critics[k], opt_a[k], opt_c[k], st, ac, lp, rt)
    m = b["exist"]                                                          # one choice sample per existing car (PY:504-507)
    n_samples += int(m.sum())
    for _ in range(10):
        PO.train_step_d(actors[2], critics[2], opt_a[2], opt_c[2], b["obs_d"][m], b["act_d"][m], b["logp_d"][m], b["rew_d"][m])
    dt = time.perf_counter() - t0
    return n_samples / dt, dt, t_roll, n_samples


def ppo_roofline(flops, tot_ms, world):
    """Useful flops of the policy MLPs (last iteration's sample counts, all ranks) over the whole iteration time,
    against the measured dense bf16 tensor throughput (the roofline the brief names for the policy GEMMs; the
    kernels compute in fp32 / 3xTF32, so three tensor-core products per useful one)."""
    peak = None
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
        src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        peak, src = 1359.2, "fallback (B200_PROFILING.md)"
    ach = flops / (tot_ms * 1e-3) / 1e12 / world
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
            "peak_source": src, "kernel": "k_ppo_grad_tc (78 % of an iteration) + k_policy_act",
            "note": "useful fp32 flops per GPU of update (54.5 kflop/sample/epoch) and rollout inference / iteration time"}


def bind_to_gpu_numa_node(torch, local):
    """Pin this rank to the CPUs of the NUMA node its GPU hangs off (sysfs), before any pinned buffer is allocated, so
    the host side of the end-to-end copies is node-local (at 8 ranks the host memory system is the e2e ceiling)."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return {"numa_node": None}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus_bound": len(cpus)}
    except Exception as e:   # no sysfs / no permission: run unbound
        return {"numa_node": None, "note": type(e).__name__}


def run_ppo(mh, torch, dist, world, rank, dev, n_envs, iters, warm=2, wl=("coop_scalable", 4, 3, 2), dump_dir=None):
    """PPO samples/s (BASELINE.json metric, second half): one iteration = one 80-step episode in every env
    (Env_rollout.iterations_rand) + reward-to-go + 10 x (cross, wait) + 10 x choice update epochs (Algo_PPO.train).
    dump_dir: rank 0 writes the last iteration's rollout buffers (sampled envs) and the six updated networks there."""
    variant, nb_car, nb_ped, nb_lines = wl
    env = mh.VecCrosswalkEnv(variant, n_envs, nb_car=nb_car, nb_ped=nb_ped, nb_lines=nb_lines, seed=1234, env_id0=rank * n_envs, device=dev)
    torch.manual_seed(0)
    C_slots = env.n_slots
    D = 2 + (6 if variant == "coop_scalable" else 5) * (C_slots - 1) + 10
    algo = mh.Algo_PPO(mh.Model_PPO, env, num_states_c=13, num_states_d=D, num_actions=1, mean=-1.0, std=3.0, nb_cars=nb_car, dt=0.3)
    r = algo.rollout
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for _ in range(warm):      # (the second identical rollout call captures and instantiates the CUDA graph the later ones replay)
        r.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        algo.update()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    n0 = mh.launch_count()
    t_roll = t_upd = 0.0
    samples = 0
    for _ in range(iters):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        r.iterations_rand(algo.actor_net_cross, algo.actor_net_wait, algo.actor_net_choice)
        e1.record()
        algo.update()
        e2.record()
        torch.cuda.synchronize()
        t_roll += e0.elapsed_time(e1); t_upd += e1.elapsed_time(e2)
        samples += sum(r.counts())
    launches = mh.launch_count() - n0
    if dump_dir and rank == 0:
        idx = torch.as_tensor(dump_envs(n_envs, DUMP_ENVS["ppo"]), device=dev)
        T, Cn = r.T, r.C
        # sample s = (t*C + car)*N + env of the [S] buffers, m = car*N + env of the [M] ones
        out = {"ppo_" + k: getattr(r, k).view(*getattr(r, k).shape[:-1], T, Cn, n_envs)[..., idx]
               for k in ("obs_c", "act", "logp", "rew", "rl", "rtg", "V")}
        out.update({"ppo_" + k: getattr(r, k).view(*getattr(r, k).shape[:-1], Cn, n_envs)[..., idx]
                    for k in ("obs_d", "act_d", "logp_d", "rew_d", "V_d")})
        out.update(ppo_route=r.route[:, idx], ppo_exist=r.exist[:, idx])
        # the networks as state_dict() hands them out (the reference's layout, not the kernels' padded one), concatenated
        out.update({"ppo_%s_%s_params" % (kind, name): torch.cat([v.reshape(-1) for v in net.state_dict().values()])
                    for name, kind, net in algo._nets()})
        write_dump(dump_dir, out)
    # useful flops of the policy networks (SURVEY.md 8d): forward 2*(D*32 + 32*64 + 64*32 + 32*out), backward = 2 x forward
    fwd = lambda D, out: 2.0 * (D * 32 + 32 * 64 + 64 * 32 + 32 * out)
    n_c, n_w, n_d = [float(x) for x in r.counts()]
    ped_mean = float(env.get_state()["env_i"][:, 1].float().mean().item())       # existing pedestrians per env (current episode)
    fl_update = 10.0 * ((n_c + n_w) * 3.0 * 2.0 * fwd(13, 1) + n_d * 3.0 * (fwd(D, 2) + fwd(D, 1)))
    pairs = C_slots * (ped_mean if variant == "coop_scalable" else nb_ped)     # the older drivers visit every pedestrian slot
    fl_roll = n_envs * (80.0 * pairs * fwd(13, 1) + C_slots * nb_ped * fwd(D, 2))
    t = torch.tensor([t_roll + t_upd, t_roll, t_upd, float(samples), fl_update + fl_roll], dtype=torch.float64, device=dev)
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX); dist.all_reduce(t, op=dist.ReduceOp.SUM)
        tot_ms, roll_ms, upd_ms, samples, flops = mx[0].item(), mx[1].item(), mx[2].item(), t[3].item(), t[4].item() * iters
    else:
        tot_ms, roll_ms, upd_ms, samples, flops = [x.item() for x in t]
        flops *= iters
    del algo, env
    torch.cuda.empty_cache()
    return {"samples_per_s": samples / (tot_ms * 1e-3), "unit": "PPO samples/s (cross + wait + choice samples consumed by the update)",
            "iteration_ms": tot_ms / iters, "rollout_ms": roll_ms / iters, "update_ms": upd_ms / iters, "iterations": iters,
            "samples_per_iteration": samples / iters, "n_envs_per_gpu": n_envs, "update_epochs": "10 x (cross, wait) + 10 x choice",
            "gpu_launches": int(launches),
            "roofline": ppo_roofline(flops, tot_ms, world),
            "config": "%s on Env_hybrid_multi_%s nb_car=%d nb_ped=%d nb_lines=%d, %d envs/GPU x 80 steps (rollout loop replayed as a CUDA graph)" % (
                {"coop_scalable": "Coop-MH-PPO-scalable", "coop": "Coop-MH-PPO.ipynb", "naif": "MH-PPO.ipynb"}.get(variant, "PPO"), variant,
                nb_car, nb_ped, nb_lines, n_envs)}


def workload_config(variant, nb_car, nb_ped, nb_lines, n_envs, state_bytes=None, flushed=True):
    """`config` of the JSON line -- the same dict for both arms (the driver compares them)."""
    if state_bytes is None:
        C = 2 * nb_lines if variant == "coop_scalable" else (2 * nb_car if "4cars" in variant else nb_car)
        state_bytes = 32 * C + 48 * nb_ped + 16
    return {"workload": "Env_hybrid_multi_%s nb_car=%d nb_ped=%d nb_lines=%d, %d envs/GPU, env.step with auto-reset, "
                        "acc ~ U(-4,2) per step, lights held per episode" % (variant, nb_car, nb_ped, nb_lines, n_envs),
            "l2": "GPU arm: flushed, an untimed 256 MiB memset (2x the 126 MB L2) runs between timed steps; the per-step working set "
                  "is ~150 MB" if flushed else "GPU arm: not flushed",
            "state_bytes_per_env": state_bytes, "parallelism": "env shards per rank, no data-path collective"}


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is single-process Python and
    cannot travel to the GPU box; this arm times its pinned C restatement (oracle/mhppo_oracle.c) on all host threads,
    on the SAME workload, warm-up and step count as the GPU arm (whole batch per step, same window of the episode)."""
    variant, nb_car, nb_ped, nb_lines, n_envs = wl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    W, K = max(args.warmup, 3), args.steps
    rate, timed, active, rounds = cpu_port_run(variant, nb_car, nb_ped, nb_lines, n_envs, W, K, threads=cores, min_seconds=5.0)
    sample = "%d envs x %d steps after %d warm-up steps, %d round(s) from a fresh reset (%.1f s timed), C oracle port " \
             "(oracle/mhppo_oracle.c), %d threads" % (n_envs, K, W, rounds, timed, cores)
    val = rate * active
    line = {"metric": "agent-steps/sec (env.step)", "value": val, "unit": "agent-steps/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * timed / (K * rounds),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(variant, nb_car, nb_ped, nb_lines, n_envs, flushed=not args.no_flush),
            "env_steps_per_s": rate, "active_agents_per_env": active, "rounds": rounds,
            "cpu_baseline": {"value": val, "unit": "agent-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "the reference is single-process Python (one env, global RNG, GIL) and is not shippable to the GPU box; "
                    "this arm is its pinned C restatement on all host threads, far faster than the Python original "
                    "(3.4k env-steps/s/core, BASELINE.md section 2)"}
    emit(line)


_JSON_FD = None


def claim_stdout():
    """Libraries (NCCL's version banner, torchrun) write to file descriptor 1; the contract is ONE JSON line on stdout.
    Everything else is sent to stderr and the line is written to the original descriptor at the end."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=160)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="scalable_432", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--per-step", action="store_true", help="add the device time of every timed step to the JSON line (profile of an episode)")
    ap.add_argument("--ppo-envs", type=int, default=131072, help="envs per GPU of the PPO samples/s section (0 = skip)")
    ap.add_argument("--ppo-iters", type=int, default=2)
    ap.add_argument("--row-major-actions", action="store_true", help="device-resident actions as a contiguous [N, A] tensor (gym layout)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (and of the last PPO iteration) "
                                                          "as DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    wl = list(WORKLOADS[args.workload])
    if args.envs:
        wl[4] = args.envs
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    if args.impl == "reference":
        return run_reference(args, wl)
    variant, nb_car, nb_ped, nb_lines, n_envs = wl

    import torch
    import torch.distributed as dist
    import mhppo_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    host_binding = bind_to_gpu_numa_node(torch, local) if world > 1 else {"numa_node": None, "note": "single rank: unbound"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps

    env = mhppo_b200.VecCrosswalkEnv(variant, n_envs, nb_car=nb_car, nb_ped=nb_ped, nb_lines=nb_lines,
                                     seed=1234, env_id0=rank * n_envs, device=dev, autoreset=True)
    A = env.n_action
    state_bytes, n_obs_env, n_lead_env = env.state_bytes_per_env, env.n_obs, env.n_lead
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    # synthetic actions resident in HBM (SURVEY.md 8d): acc ~ U(-4,2) fresh every step (4 draws, cycled), light in {-1,+1}
    # drawn once per episode and held (2 light draws, alternating from one 80-step episode to the next)
    lights = [(torch.rand(n_envs, A // 2, device=dev, generator=g) < 0.5).float() * 2 - 1 for _ in range(2)]
    acts = []
    for e in range(2):
        row = []
        for _ in range(4):
            # [N, A] view of a component-major buffer: the layout the rollout kernels hand to env.step (coalesced reads)
            a = torch.empty(n_envs, A, device=dev) if args.row_major_actions else torch.empty(A, n_envs, device=dev).t()
            a[:, :A // 2] = torch.rand(n_envs, A // 2, device=dev, generator=g) * 6 - 4
            a[:, A // 2:] = lights[e]
            row.append(a)
        acts.append(row)
    pick = lambda lst, t: lst[(t // EPISODE) % 2][t % 4]      # t = steps since the reset
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    env.reset()
    for t in range(W):
        env.step(pick(acts, t))
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed region: K steps, one event pair per step, L2 flushed between steps -----------
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    n0 = mhppo_b200.launch_count()
    wall0 = time.perf_counter()
    for t in range(K):
        if flush is not None:
            flush.zero_()
        ev[t][0].record()
        last = env.step(pick(acts, W + t))
        ev[t][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    launches = mhppo_b200.launch_count() - n0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = sum(step_ms)
    if args.dump_outputs and rank == 0:          # before the end-to-end region steps the same envs further
        obs, rew, done, trunc, _ = last
        idx = torch.as_tensor(dump_envs(n_envs, DUMP_ENVS["env_step"]), device=dev)
        out = {"env_step_obs_" + k: v[idx] for k, v in obs.items()}
        out.update(env_step_rewards=rew[idx], env_step_done=done[idx], env_step_truncated=trunc[idx],
                   env_step_reward_light=env.reward_light[idx], env_step_terminal_obs=env.terminal_obs[idx])
        write_dump(args.dump_outputs, out)

    # ---- end-to-end region: host buffers through the reference-facing call -------------------------
    Ke = max(8, min(K, 40))
    act_h = [[p.cpu().pin_memory() for p in row] for row in acts]
    obs_h = torch.empty(n_envs, env.n_obs).pin_memory()
    rew_h = torch.empty(n_envs, env.n_lead).pin_memory()
    rl_h = torch.empty(n_envs, env.n_lead).pin_memory()
    done_h = torch.empty(n_envs, dtype=torch.uint8).pin_memory()
    for t in range(3):
        env.step_host(pick(act_h, W + K + t), obs_h, rew_h, rl_h, done_h)
    barrier()
    e0 = time.perf_counter()
    for t in range(Ke):
        env.step_host(pick(act_h, W + K + 3 + t), obs_h, rew_h, rl_h, done_h)
    barrier()
    e2e_s = time.perf_counter() - e0
    h2d = n_envs * A * 4
    d2h = n_envs * (n_obs_env + 2 * n_lead_env) * 4 + n_envs

    st = env.get_state()
    active = float((st["env_i"][:, 1] + st["env_i"][:, 2]).float().mean().item())
    flushed = flush is not None
    del st, env, last, flush, acts, act_h, obs_h
    torch.cuda.empty_cache()
    ppo = None
    if args.ppo_envs > 0 and args.ppo_iters > 0:
        if args.workload == "scalable_432":
            ppo = run_ppo(mhppo_b200, torch, dist, world, rank, dev, args.ppo_envs, args.ppo_iters, dump_dir=args.dump_outputs)
        elif variant in ("coop", "naif", "stop"):       # the older drivers' PPO on their own env class, at the workload's env count
            ppo = run_ppo(mhppo_b200, torch, dist, world, rank, dev, n_envs, max(args.ppo_iters, 5), warm=3, wl=(variant, nb_car, nb_ped, nb_lines),
                          dump_dir=args.dump_outputs)
    clocks = sampler.stop()        # sampled every 200 ms from the start of the device-timed region to the end of the PPO section
    t_dev = torch.tensor([dev_ms, e2e_s, active], dtype=torch.float64, device=dev)
    if world > 1:
        mx = t_dev.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_dev, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, active = mx[0].item(), mx[1].item(), t_dev[2].item() / world

    if rank == 0:
        B, C, nobs = algorithmic_bytes(variant, nb_car, nb_ped, nb_lines)
        peak, peak_src = measured_peaks()
        env_steps = world * n_envs * K / (dev_ms * 1e-3)
        kern_ms = dev_ms / K
        achieved = B * n_envs / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": "agent-steps/sec (env.step)", "value": env_steps * active, "unit": "agent-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": kern_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(variant, nb_car, nb_ped, nb_lines, n_envs, state_bytes, flushed),
            "env_steps_per_s": env_steps, "slot_agent_steps_per_s": env_steps * (C + nb_ped),
            "active_agents_per_env": active, "wall_s_timed_region": wall, "gpu_launches": int(launches),
            "clocks": clocks, **({"per_step_ms": [round(x, 5) for x in step_ms]} if args.per_step else {}),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": recorded_traffic(n_envs)[0] if args.workload == "scalable_432" else None,
                         "traffic_source": recorded_traffic(n_envs)[1] if args.workload == "scalable_432" else None,
                         "algorithmic_bytes_per_env_step": B, "peak_source": peak_src,
                         "kernel": "k_env_step<%s>" % variant},
            "e2e": {"value": world * n_envs * Ke / e2e_s * active, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": Ke, "pcie_gbs_per_gpu": (h2d + d2h) * Ke / e2e_s / 1e9, "host_binding": host_binding,
                    "call": "mhppo_env_step_host (pinned host buffers; env range in slices over 3 streams: H2D, kernel and D2H overlap)"},
        }
        if ppo is not None:
            line["ppo"] = ppo
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            # the same procedure as `--impl reference`: whole batch, same warm-up and window, >= 10 s of timed CPU work
            rate, dt, act_cpu, rounds = cpu_port_run(variant, nb_car, nb_ped, nb_lines, n_envs, W, K, threads=cores, min_seconds=10.0)
            line["cpu_baseline"] = {"value": rate * act_cpu, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                                    "sample": "%d envs x %d steps after %d warm-up steps, %d round(s) from a fresh reset (%.1f s timed), "
                                              "C oracle port on all host threads" % (n_envs, K, W, rounds, dt),
                                    "env_steps_per_s": rate}
            if ppo is not None:
                n_cpu = 256
                r_ppo, dt_ppo, dt_roll, n_s = cpu_ppo_rate(n_cpu, (variant, nb_car, nb_ped, nb_lines) if args.workload != "scalable_432" else ("coop_scalable", 4, 3, 2))
                ppo["cpu_baseline"] = {"value": r_ppo, "unit": "PPO samples/s", "cores": cores, "kind": "port",
                                       "sample": "one iteration at %d envs (%d samples, %.1f s of which rollout %.1f s): vectorised numpy/torch "
                                                 "restatement of Env_rollout + Algo_PPO (oracle/ppo_oracle.py) over the C env port; the "
                                                 "unmodified per-sample Python reference does 544 samples/s (BASELINE.md section 2)" % (
                                                     n_cpu, n_s, dt_ppo, dt_roll)}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
