"""Learning-curve reproduction (SURVEY.md 8 f2): Algo_PPO.train on the scalable 1/1/1 config -- the only configuration the
reference publishes curves for (load_model/parameters/pappo-scalable-coop-111-*-step-001000.npy, written by PY:908-916).

  python tools/train_curves.py --envs 26 --iters 1000 --out profiles/round2_learning/n26      # 26 envs = the reference's 2080 samples / iteration
  python tools/train_curves.py --envs 4096 --iters 300 --out profiles/round2_learning/n4096   # one large-N run
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --minibatches 8 --out ...      # B = 8 shuffled minibatches per epoch
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --diagnostics --entropy-coef 0.01 --out ...   # update diagnostics
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --max-grad-norm 0.5 --out ...   # per-net gradient-norm clipping
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --lr-schedule adaptive --desired-kl 0.01 --out ...   # KL-adaptive lr
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --lr-schedule linear --lr-anneal-iterations 300 --out ...
  python tools/train_curves.py --envs 4096 --iters 300 --seed 4 --normalize-reward --max-grad-norm inf --out ...   # reward scaling

Writes the four traces with the reference's file names under <out>/load_model/parameters/, the checkpoints under
<out>/load_model/weights/, <out>/summary.json (means of the first / last 10 iterations, wall time) and <out>/traces.json
(the four traces as text; with --diagnostics or --target-kl also the per-iteration update diagnostics of each pair,
Algo_PPO.ep_diagnostics, as traces "diag_<pair>_<field>"; with --max-grad-norm the per-iteration mean gradient norms of each
pair, Algo_PPO.ep_grad_norms, as traces "gradnorm_<pair>_<field>"; with --lr-schedule each pair's lrs after every update,
Algo_PPO.ep_lrs, as traces "lr_<pair>_<actor_lr|critic_lr>"; with --normalize-reward the running reward statistics after every
update, Algo_PPO.ep_reward_norm, as traces "rewnorm_<continuous|choice>_<count|mean|var|scale>")."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mhppo_b200  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=26)
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=10)
    ap.add_argument("--out", default="profiles/round2_learning/n26")
    ap.add_argument("--minibatches", type=int, default=None, help="Algo_PPO(n_minibatches=B); default: full-batch epochs")
    ap.add_argument("--diagnostics", action="store_true", help="Algo_PPO(diagnostics=True): per-iteration update diagnostics")
    ap.add_argument("--target-kl", type=float, default=None, help="Algo_PPO(target_kl=delta): halt a pair's update at approx. KL > 1.5 delta")
    ap.add_argument("--entropy-coef", type=float, default=0.0, help="Algo_PPO(entropy_coef=c): entropy bonus of the choice actor")
    ap.add_argument("--max-grad-norm", type=float, default=None, help="Algo_PPO(max_grad_norm=g): clip each net's gradient norm to g")
    ap.add_argument("--lr-schedule", choices=["linear", "adaptive"], default=None, help="Algo_PPO(lr_schedule=...)")
    ap.add_argument("--desired-kl", type=float, default=None, help="Algo_PPO(desired_kl=delta): the adaptive schedule's KL target")
    ap.add_argument("--lr-anneal-iterations", type=int, default=None, help="Algo_PPO(lr_anneal_iterations=K): the linear schedule's length")
    ap.add_argument("--normalize-reward", action="store_true", help="Algo_PPO(normalize_reward=True): SB3's reward scaling")
    ap.add_argument("--clip-reward", type=float, default=None, help="Algo_PPO(clip_reward=c): clip of the scaled rewards (default 10)")
    ap.add_argument("--car", type=int, default=1); ap.add_argument("--ped", type=int, default=1); ap.add_argument("--lines", type=int, default=1)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    env = mhppo_b200.VecCrosswalkEnv("coop_scalable", a.envs, nb_car=a.car, nb_ped=a.ped, nb_lines=a.lines, seed=a.seed)
    torch.manual_seed(a.seed)
    D = 2 + 6 * (2 * a.lines - 1) + 10
    algo = mhppo_b200.Algo_PPO(mhppo_b200.Model_PPO, env, num_algo=100 * a.ped + 10 * a.car + a.lines, num_states_c=13, num_states_d=D,
                               num_actions=1, mean=-1.0, std=3.0, nb_cars=a.car, dt=0.3, n_minibatches=a.minibatches,
                               diagnostics=a.diagnostics, target_kl=a.target_kl, entropy_coef=a.entropy_coef,
                               max_grad_norm=a.max_grad_norm, lr_schedule=a.lr_schedule, desired_kl=a.desired_kl,
                               lr_anneal_iterations=a.lr_anneal_iterations, normalize_reward=a.normalize_reward,
                               clip_reward=a.clip_reward)
    t0 = time.perf_counter()
    algo.train(a.iters, root=a.out)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    algo.saving(root=a.out)
    m = lambda x, s: float(np.mean(x[s])) if len(x) else None
    summ = {"envs": a.envs, "iterations": a.iters, "config": "%d/%d/%d" % (a.ped, a.car, a.lines), "wall_s": wall,
            "samples_per_iteration_mean": float(np.mean(np.sum(algo.ep_scenario_balance, axis=1))),
            "reward_cross_first10": m(algo.ep_reward_cross, slice(0, 10)), "reward_cross_last10": m(algo.ep_reward_cross, slice(-10, None)),
            "reward_wait_first10": m(algo.ep_reward_wait, slice(0, 10)), "reward_wait_last10": m(algo.ep_reward_wait, slice(-10, None)),
            "reward_choice_first10": m(algo.ep_reward_choice, slice(0, 10)), "reward_choice_last10": m(algo.ep_reward_choice, slice(-10, None)),
            "reward_cross_last": algo.ep_reward_cross[-1] if algo.ep_reward_cross else None,
            "scenario_balance_last": [int(v) for v in algo.ep_scenario_balance[-1]],
            "scenario_balance_last10_mean": [float(v) for v in np.mean(algo.ep_scenario_balance[-10:], axis=0)],
            "n_minibatches": a.minibatches, "diagnostics": a.diagnostics, "target_kl": a.target_kl, "entropy_coef": a.entropy_coef, "max_grad_norm": a.max_grad_norm,
            "lr_schedule": a.lr_schedule, "desired_kl": a.desired_kl, "lr_anneal_iterations": a.lr_anneal_iterations,
            "normalize_reward": a.normalize_reward, "clip_reward": a.clip_reward, "seed": a.seed, "mlp_mode": os.environ.get("MHPPO_MLP", "auto")}
    json.dump(summ, open(os.path.join(a.out, "summary.json"), "w"), indent=1)
    traces = {"reward_cross": algo.ep_reward_cross, "reward_wait": algo.ep_reward_wait, "reward_choice": algo.ep_reward_choice,
              "scenario_balance": [[int(v) for v in r] for r in algo.ep_scenario_balance]}
    for it in algo.ep_diagnostics:
        for p, d in it.items():
            for k, v in d.items():
                traces.setdefault("diag_%s_%s" % (p, k), []).append(v)
    for it in algo.ep_grad_norms:
        for p, d in it.items():
            for k, v in d.items():
                traces.setdefault("gradnorm_%s_%s" % (p, k), []).append(v)
    for it in algo.ep_lrs:
        for p, d in it.items():
            for k, v in d.items():
                traces.setdefault("lr_%s_%s" % (p, k), []).append(v)
    for it in algo.ep_reward_norm:
        for p, d in it.items():
            for k, v in d.items():
                traces.setdefault("rewnorm_%s_%s" % (p, k), []).append(v)
    json.dump(traces, open(os.path.join(a.out, "traces.json"), "w"))             # the .npy traces as text
    print(json.dumps(summ))


if __name__ == "__main__":
    main()
