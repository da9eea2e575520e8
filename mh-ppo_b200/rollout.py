"""Env_rollout -- vectorised mirror of the reference's rollout class (Coop-MH-PPO-scalable.py:96-684)
for the scalable env class: every env runs one 80-step episode per call, the per-(car, pedestrian)
feature builders, policy inference, sampling, log-probs and buffer writes run in the kernels of
libmhppo_b200.so, and the env-step kernel writes rewards / reward_light straight into the rollout
buffers (zero copy).

Buffers (CUDA, fp32, env index innermost; include/mhppo.h "Buffers"):
  obs_c [13][S], act/logp/rew/rl/rtg [S] with S = T*C*N and sample s = (t*C + car)*N + env
  obs_d [D][M], act_d/logp_d/rew_d [M] with M = C*N;   route int8 [C][N]: 0 cross, 1 wait, -1 car absent
"""
import ctypes as C

import torch

from . import _lib
from ._lib import RolloutCfg, View, check


class Env_rollout:
    def __init__(self, env, nb_cars, max_steps, dt, seed=None):
        # scalable: Coop-MH-PPO-scalable.py.  coop / naif / stop (6-float car rows, 3-float env row): the two older drivers,
        # Coop-MH-PPO.ipynb (coop) and MH-PPO.ipynb (naif), whose PPO cells are identical ("legacy" feature layout)
        if env.variant not in ("coop_scalable", "coop", "naif", "stop"):
            raise NotImplementedError("no PPO driver of the reference runs on the %s env class (its observation has the extra "
                                      "car_follow key)" % env.variant)
        self.legacy = env.variant != "coop_scalable"
        self.env, self.nb_cars, self.max_steps, self.dt = env, nb_cars, max_steps, dt
        self._L = _lib.lib()
        N, Cn, P, T = env.n_envs, env.n_slots, env.nb_ped, max_steps
        self.N, self.C, self.P, self.T = N, Cn, P, T
        self.shape_env = 2 + 9 + 2                       # PY:110
        self.shape_env_d = 2 + (5 if self.legacy else 6) * (Cn - 1) + 8 + 2      # PY:111 / NB2 cell 1 (5 columns per other car)
        dev = env.device
        S, M = T * Cn * N, Cn * N
        self.S, self.M = S, M
        f = lambda *s: torch.zeros(*s, device=dev)
        self.obs_c, self.act, self.logp, self.rew, self.rl, self.rtg, self.V = f(13, S), f(S), f(S), f(S), f(S), f(S), f(S)
        self.obs_d, self.act_d, self.logp_d, self.rew_d, self.V_d = f(self.shape_env_d, M), f(M), f(M), f(M), f(M)
        self.action_d = torch.zeros(Cn * P, N, dtype=torch.int8, device=dev)
        self.light = f(Cn, N)
        self.actions = f(2 * Cn, N)                      # env action buffer, component-major
        self.route = torch.zeros(Cn, N, dtype=torch.int8, device=dev)
        self.exist = torch.zeros(Cn, N, dtype=torch.int8, device=dev)
        self._cfg = RolloutCfg(nb_ped=P, nb_lines=env.nb_lines, T=T, legacy_nb_car=Cn if self.legacy else 0, n_envs=N, seed=env._seed,
                               env_id0=env._env_id0)
        self.iteration = 0
        self.use_graph = True                            # replay the T-step loop as a CUDA graph (mhppo_rollout_steps)
        self.value_std = 0.5                             # exploration variance of the Gaussian head (Algo_PPO.value_std, PY:726)
        self.ret = None                                  # GAE returns [S]: allocated by the first gae() call

    def _set_head(self, actor):
        """The kernels' Gaussian head = the actor's own (tanh * std + mean, PY:88-90), the noise variance of PY:726-729 and
        car_b[1,0] as the start of the min over pedestrians (PY:436) -- so Model_PPO.forward, rollout and update agree."""
        check(self._L.mhppo_set_gaussian_head(float(actor.mean), float(actor.std), float(self.value_std), float(self.env.car_b[1, 0])))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    def reset(self):
        """Reset (PY:125-150): a fresh episode in every env."""
        self.env.reset()

    def iterations_rand(self, actor_net_cross, actor_net_wait, actor_net_choice, cov_mat=None, cov_mat_d=None, batch_size=None,
                        random_rate=0.0):
        """One episode per env of the reference's rollout (PY:357-516).  Resets the envs first (PY:377)."""
        env, L, cfg, st = self.env, self._L, self._cfg, self._stream()
        N, Cn, T = self.N, self.C, self.T
        if (actor_net_cross.mean, actor_net_cross.std) != (actor_net_wait.mean, actor_net_wait.std):
            raise ValueError("the cross and wait actors must share mean / std (PY:711-714)")
        self._set_head(actor_net_cross)
        env.reset()
        if self.legacy:
            self.exist.fill_(1)                          # every car exists in the older drivers (no cars_exist test)
        else:
            self.exist.copy_(env.get_state()["car_i"][:, :, 1].t().to(torch.int8))           # cars_exist, PY:380
        check(L.mhppo_choice_act(C.byref(cfg), env._obs.data_ptr(), actor_net_choice.flat.data_ptr(), self.iteration,
                                 self.action_d.data_ptr(), self.light.data_ptr(), self.obs_d.data_ptr(), self.act_d.data_ptr(),
                                 self.logp_d.data_ptr(), st))
        # the T-step loop (policy_act -> env.step, no auto-reset: the episode ends exactly at step T-1; the next call resets)
        # runs inside the library: one call, replayed as a CUDA graph from the second iteration on
        check(L.mhppo_rollout_steps(env._h, C.byref(cfg), env._obs.data_ptr(), actor_net_cross.flat.data_ptr(),
                                    actor_net_wait.flat.data_ptr(), self.action_d.data_ptr(), self.light.data_ptr(), self.iteration,
                                    self.actions.data_ptr(), self.obs_c.data_ptr(), self.act.data_ptr(), self.logp.data_ptr(),
                                    self.rew.data_ptr(), self.rl.data_ptr(), env._done.data_ptr(), int(self.use_graph), st))
        # trajectory routing (PY:489-502): existing car i goes to the cross buffer if action_d[i] <= 0, where i indexes the
        # flat (car x ped) decision array -- the reference's own quirk (SURVEY.md hard part 6) -- else to the wait buffer
        flat_d = self.action_d[:Cn]                      # rows 0..C-1 of the (car*P + ped) array
        self.route.copy_(torch.where(self.exist != 0, (flat_d > 0).to(torch.int8), torch.full_like(flat_d, -1)))
        self.iteration += 1

    def choix_test(self):
        """The fixed test scenario of the reference (PY:629-633): pedestrian 0 at (0, -1) walking at 1.25 m/s, car 0 at -45 m
        in lane 0 and car 1 at -22 m in lane 1, both keeping their speed.  As under gym 0.26 (whose wrappers do not forward
        attribute writes) `self.env.cross = 3.` does not reach the env: the crossing width stays the episode's."""
        env = self.env
        v = env.flat_obs[:, 1].clone()                        # self.env.state["car"][1]
        env.reset_pedestrian(0, 0.0, 1.25, 0.0, -1.0, 0, -1, 3.0, True, 1)
        env.reset_cars(0, v, -45.0, 0.0, 0.0)
        if env.n_slots > 1:
            env.reset_cars(1, v, -22.0, 0.0, 1.0)
        return env.observe()                                  # state = self.env.get_state(), PY:173

    def iterations_dataset(self, actor_net_cross, actor_net_wait, actor_net_choice, snapshot, **kw):
        """Env_rollout.iterations_dataset (PY:255-355): one deterministic evaluation episode from every scenario of a stored
        dataset.  The reference unpickles a list of deep-copied envs (`test_data_23.pickle`, not shipped); here the dataset
        is a snapshot file of VecCrosswalkEnv.save_state (one scenario per env)."""
        self.env.load_state(snapshot)
        return self.iterations(actor_net_cross, actor_net_wait, actor_net_choice, 1, start="current", **kw)

    def iterations(self, actor_net_cross, actor_net_wait, actor_net_choice, nbr_episodes, choix=False, record_obs=True,
                   record_waiting=True, start="reset"):
        """Deterministic evaluation rollout (PY:152-252): `nbr_episodes` episodes in every env, argmax decisions (re-taken
        every step while ped_traffic != nb_ped), accelerations = min over all pedestrian slots of the cross / wait net or
        the speed-recovery action, capped by (10 - v)/dt.  Returns a dict of CUDA tensors, episode-major:
          obs [E,T,n_obs,N] (state before each step), acts [E,T,C,N], rews [E,T,C,N], reward_light [E,T,C,N],
          action_d int8 [E,T,C*P,N] (+-1 decisions in force at each step), waiting [E,T,P,N] (pedestrian.waiting_time
          after each step).  `reference_batches(out, n)` rebuilds the reference's return values for env n."""
        if self.legacy:
            raise NotImplementedError("the deterministic evaluation rollout is built for Coop-MH-PPO-scalable.py only")
        env, L, cfg, st = self.env, self._L, self._cfg, self._stream()
        N, Cn, P, T, dev = self.N, self.C, self.P, self.T, env.device
        self._set_head(actor_net_cross)
        E = int(nbr_episodes)
        f = lambda *s: torch.zeros(*s, device=dev)
        out = dict(acts=f(E, T, Cn, N), rews=f(E, T, Cn, N), reward_light=f(E, T, Cn, N),
                   action_d=torch.zeros(E, T, Cn * P, N, dtype=torch.int8, device=dev))
        if record_obs:
            out["obs"] = f(E, T, env.n_obs, N)
        if record_waiting:
            out["waiting"] = f(E, T, P, N)
        was_auto = env.autoreset
        env.autoreset = False
        none = View(None, 0, 0)
        lo, hi = float(env.car_b[0, 0]), float(env.car_b[1, 0])
        for e in range(E):
            if start == "current" and e == 0:
                env.observe()                            # state = self.env.get_state(), PY:275
            else:
                env.reset()
                if choix:
                    self.choix_test()                    # PY:171-173
            for t in range(T):
                check(L.mhppo_choice_eval(C.byref(cfg), env._obs.data_ptr(), actor_net_choice.flat.data_ptr(), int(t == 0),
                                          self.action_d.data_ptr(), st))
                if record_obs:
                    out["obs"][e, t].copy_(env._obs)
                out["action_d"][e, t].copy_(self.action_d)
                check(L.mhppo_policy_eval(C.byref(cfg), env._obs.data_ptr(), actor_net_cross.flat.data_ptr(),
                                          actor_net_wait.flat.data_ptr(), self.action_d.data_ptr(), float(self.dt),
                                          float(env.speed_limit), lo, hi, self.actions.data_ptr(), out["acts"][e, t].data_ptr(), st))
                check(L.mhppo_env_step(env._h, View(self.actions.data_ptr(), 1, N), View(env._obs.data_ptr(), 1, N),
                                       View(out["rews"][e, t].data_ptr(), 1, N), View(out["reward_light"][e, t].data_ptr(), 1, N),
                                       env._done.data_ptr(), 0, none, st))
                if record_waiting:
                    out["waiting"][e, t].copy_(env.ped_waiting_time.t())
        env.autoreset = was_auto
        return out

    def reference_batches(self, out, n):
        """The reference's return values of `iterations` (PY:238-252) for env `n`, rebuilt from the dense records:
        (t_batch_obs, t_batch_acts, t_batch_rews_c, t_batch_rews_d, t_batch_waiting_time) as CPU tensors.  The reference
        closes a batch after every step while ped_traffic != nb_ped (episodic reward = min(0, reward_light) of that one
        step, PY:222-235) and once per episode otherwise (min over the episode)."""
        E, T = out["acts"].shape[:2]
        Cn, P = self.C, self.P
        obs = out["obs"][:, :, :, n].reshape(E * T, -1).cpu()
        acts = out["acts"][:, :, :, n].reshape(E * T, Cn).cpu()
        rews_c = out["rews"][:, :, :, n].reshape(E * T, Cn).cpu()
        rl = out["reward_light"][:, :, :, n].cpu()
        wait = out["waiting"][:, :, :, n].cpu()
        rews_d, wt = [], []
        for e in range(E):
            per_step = float(out["obs"][e, 0, 7 * Cn + 1, n]) != float(P)           # ped_traffic is fixed during an episode
            if per_step:
                rews_d.append(torch.minimum(rl[e], torch.zeros_like(rl[e])))
                wt.append(wait[e].reshape(-1))
            else:
                rews_d.append(torch.minimum(rl[e].min(dim=0).values, torch.zeros(Cn))[None])
                wt.append(wait[e, T - 1])
        return obs, acts, rews_c, torch.cat(rews_d), torch.cat(wt)

    def get_average(self, out):
        """The reference's episode statistics (analysis cell `get_average`, PY:1550-1675; waiting-time histogram input
        PY:1390-1403) of an evaluation record `out` = iterations(...), computed on the device: one kernel walks every
        (episode, env) record once (mhppo_episode_stats), the means / standard deviations / scenario frequencies are torch
        reductions of its per-episode arrays.  Returns a dict with the cell's own names, plus `waiting_times` (seconds, one
        entry per episode and pedestrian slot: what the reference histograms)."""
        obs = out["obs"].contiguous()
        E, T, n_obs, N = obs.shape
        Cn, P, dev = self.C, self.P, obs.device
        cw, ew = (6, 3) if self.legacy else (7, 4)
        ped = torch.zeros(2, E, P, N, device=dev); car = torch.zeros(8, E, Cn, N, device=dev)
        sums = torch.zeros(E, N, 8, dtype=torch.float64, device=dev); ys = torch.zeros(E, N, 3, dtype=torch.float64, device=dev)
        check(self._L.mhppo_episode_stats(obs.data_ptr(), E, T, Cn, P, cw, ew, N, float(self.dt), ped.data_ptr(), car.data_ptr(),
                                          sums.data_ptr(), ys.data_ptr(), self._stream()))
        d = lambda t: t.double()

        def mstd(n, s, ss):                                   # mean and unbiased std (torch.std) from moments
            n, s, ss = float(n), float(s), float(ss)
            if n < 1:
                return float("nan"), float("nan")
            m = s / n
            return m, (max(ss - n * m * m, 0.0) / (n - 1)) ** 0.5 if n > 1 else float("nan")

        def mstd_t(x):
            x = d(x).reshape(-1)
            return (float(x.mean()) if x.numel() else float("nan")), (float(x.std()) if x.numel() > 1 else float("nan"))

        S = sums.sum(dim=(0, 1)).cpu()
        res = {}
        res["mean_speed"], res["sqrt_speed"] = mstd(S[0], S[1], S[2])
        res["mean_acc"] = float(S[3] / S[0]); res["sqrt_acc"] = mstd(S[0], S[4], S[5])[1]
        res["mean_speed_p"], res["sqrt_speed_p"] = mstd(S[0], S[6], S[7])
        Y = ys.sum(dim=(0, 1)).cpu()
        res["mean_speed_cars"], res["sqrt_speed_cars"] = mstd(Y[0], Y[1], Y[2])
        wait, pleave = ped[0], ped[1]                         # [E, P, N]
        leave, free, decision, light1, could, en, es, ess = car
        FI = torch.cat([d(pleave), d(leave)], dim=1); FN = torch.cat([d(pleave) - d(wait), d(free)], dim=1)      # [E, P + C, N]
        res["interaction_cost"] = float((FI.max(dim=1).values - FN.max(dim=1).values).mean())
        res["max_finish_compare"] = float((FI - FN).mean())
        y = light1 == 1
        res["mean_temp_cars"], res["std_temp_cars"] = mstd(d(en)[y].sum(), d(es)[y].sum(), d(ess)[y].sum())
        res["mean_all_temp_cars"], res["std_all_temp_cars"] = mstd_t(leave)
        res["mean_temp_peds"], res["std_temp_peds"] = mstd_t(pleave)
        n_ep = float(E * N)
        res["yield_decision"] = float((decision == 1).sum()) / n_ep
        res["go_first_decision"] = float((decision == -1).sum()) / n_ep
        w = d(wait).reshape(-1)
        res["mean_waiting"], res["std_waiting"] = float(w.mean()), float(w.std(unbiased=False))
        cs = could[could >= 0]
        res["could_stop"] = float(d(cs).mean()) if cs.numel() else float("nan")
        res["n_episodes"] = int(n_ep)
        if Cn == 2:
            s2 = decision.sum(dim=1)
            res["scenario_11"] = float((s2 == 2).sum()) / n_ep; res["scenario_m1m1"] = float((s2 == -2).sum()) / n_ep
            res["scenario_m11"] = float(((decision[:, 0] == -1) & (decision[:, 1] == 1)).sum()) / n_ep
            res["scenario_1m1"] = float(((decision[:, 0] == 1) & (decision[:, 1] == -1)).sum()) / n_ep
        res["waiting_times"] = wait.permute(2, 0, 1).reshape(-1)          # env-major, like back-to-back episodes of one env
        return res

    def futur_rewards(self):
        """Expected future rewards (PY:658-684) for every trajectory + the episodic choice reward (PY:461, 504)."""
        check(self._L.mhppo_returns(self.rew.data_ptr(), self.rl.data_ptr(), self.T, self.M, 0.99, self.rtg.data_ptr(),
                                    self.rew_d.data_ptr(), self._stream()))
        return self.rtg, self.rew_d

    def gae(self, critic_cross, critic_wait, gamma, lam, selections=None, workspace=None):
        """GAE(gamma, lambda) returns of the cross / wait buffers, an option of Algo_PPO (the reference's estimator is
        futur_rewards: lambda = 1 against the critic of every epoch).  Each critic evaluates V_old(s) once on the samples
        routed to its net (mhppo_value_stats, into self.V), then one reverse scan per (car, env) column (mhppo_gae) with
        V(s_T) = 0.  selections: the (idx, K) compacted column lists of route 0 and 1 (Algo_PPO._selection), built from
        `route` when None.  Returns (ret [S], stats6): the regression targets and this rank's advantage statistics
        (sum A, sum A^2, n) of the cross samples, then of the wait samples.  The buffers are allocated on the first call."""
        L, st, dev = self._L, self._stream(), self.rew.device
        if self.ret is None:
            self.ret = torch.zeros(self.S, device=dev)
            self._gae_stats = torch.zeros(9, dtype=torch.float64, device=dev)      # stats6 | scratch of mhppo_value_stats
        if workspace is None:
            if getattr(self, "_gae_ws", None) is None:
                self._gae_ws = torch.zeros(L.mhppo_update_workspace_bytes(13), dtype=torch.uint8, device=dev)
            workspace = self._gae_ws
        if selections is None:
            selections = []
            for want in (0, 1):
                sel = torch.nonzero(self.route.view(-1) == want).view(-1).to(torch.int32)
                selections.append((sel if sel.numel() else torch.zeros(1, dtype=torch.int32, device=dev), sel.numel()))
        ws, scratch = workspace.data_ptr(), self._gae_stats.data_ptr() + 6 * 8
        for critic, (idx, K) in zip((critic_cross, critic_wait), selections):
            check(L.mhppo_value_stats(13, self.obs_c.data_ptr(), 13, self.S, idx.data_ptr(), K, self.M, critic.flat.data_ptr(),
                                      self.rew.data_ptr(), self.V.data_ptr(), scratch, ws, st))
        check(L.mhppo_gae(self.rew.data_ptr(), self.V.data_ptr(), self.route.data_ptr(), self.T, self.M, float(gamma), float(lam),
                          self.ret.data_ptr(), self._gae_stats.data_ptr(), ws, st))
        return self.ret, self._gae_stats[:6]

    def counts(self):
        """(cross, wait, choice) sample counts of the last rollout."""
        ncross = int((self.route == 0).sum().item()) * self.T
        nwait = int((self.route == 1).sum().item()) * self.T
        return ncross, nwait, int((self.exist != 0).sum().item())

    def immediate_rewards(self):
        """Mean immediate rewards per buffer (PY:635-656, reduced on device)."""
        r = self.rew.view(self.T, self.C, self.N)
        mc, mw = (self.route == 0), (self.route == 1)
        cross = r[:, mc].mean() if mc.any() else None
        wait = r[:, mw].mean() if mw.any() else None
        choice = self.rew_d.view(self.C, self.N)[self.exist != 0].mean()
        return cross, wait, choice
