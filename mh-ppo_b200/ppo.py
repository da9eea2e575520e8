"""Algo_PPO -- vectorised mirror of the reference's PPO class (Coop-MH-PPO-scalable.py:698-1001) for the
scalable env class: same constructor (`Algo_PPO(policy_class, env, **hyperparameters)`), same six networks
and six Adam optimisers, same update rule (clipped surrogate 0.8/1.2, no entropy term, MSE critic, 10 full-batch
epochs per net per iteration, advantages = reward-to-go - V normalised with the unbiased std).

Two options beyond the reference, both off by default (DESIGN.md §4 "GAE and entropy options"):
  gae_lambda=None   a number in [0, 1]: the cross / wait nets train on GAE(gamma, lambda) returns and advantages, formed
                    once per update from the critics before the update (Env_rollout.gae); the choice net is unchanged
  entropy_coef=0.0  c > 0: the choice actor's loss gets the entropy bonus -c * mean_s H(pi(.|s))
A third option, also off by default (DESIGN.md §4 "Minibatches"):
  n_minibatches=None  an integer B in [1, 1024]: every epoch splits each net's columns ((car, env) trajectories) into B
                    shuffled minibatches and takes one Adam step per minibatch instead of one full-batch step.  The buckets
                    come from Philox stream 3 (mhppo_minibatch_plan), identical for any number of ranks; a minibatch with
                    fewer than 2 samples over all ranks takes no step.  The unused `batch_size` of the reference stays unused.
Two more, also off by default (DESIGN.md §4 "Diagnostics"):
  diagnostics=False   True: every Adam step of an update gets a record (approx. KL, clip fraction, choice entropy, explained
                      variance, both losses), computed on the device in the step's gradient pass; update() leaves them in
                      `last_update_stats`, train() appends per-iteration means to `ep_diagnostics`.  No weight bit changes.
  target_kl=None      delta > 0: a pair takes no further step in an update once a step's approx. KL exceeds 1.5 delta (SB3's
                      rule, checked on the device before the step, no host round trip).  Turns the diagnostics on.
One more, also off by default (DESIGN.md §5 "Gradient-norm clipping"):
  max_grad_norm=None  g > 0 (+inf allowed): before each Adam step, each of the six nets' gradients is clipped on its own, as
                      torch.nn.utils.clip_grad_norm_(net.parameters(), g) would before that net's optimiser step: with norm = the L2
                      norm of the net's whole all-reduced gradient, the step uses g / (norm + 1e-6) * grad when that factor is < 1.
                      A non-finite norm leaves the step unclipped; g = inf never clips.  Fused into the pair's Adam launch
                      (mhppo_adam2_clip).  update() leaves every step's two norms in `last_grad_norms`, train() appends
                      per-iteration means to `ep_grad_norms`.
A learning-rate schedule, also off by default (DESIGN.md §4 "Learning-rate schedules", §5 "Learning-rate schedule cost"):
  lr_schedule=None    every lr stays what its Adam holds (the constructor's actor_lr / critic_lr / actor_d_lr / critic_d_lr).
  "linear"            with lr_anneal_iterations=K (an integer >= 1): at the start of every update() each of the six optimisers gets
                      lr = lr0 * max(0, 1 - k / K), lr0 its constructor value and k = self.total_loop, the iterations train() has
                      completed (loading() sets it too); CleanRL's anneal_lr.  Host only: the steps take the usual Adam launches.
  "adaptive"          with desired_kl=delta (a finite number > 0): rsl_rl's schedule="adaptive" rule, decided on the device before
                      every step of a pair (each full-batch epoch, each minibatch that takes a step): kl = the step's approx. KL (the
                      all-reduced k3 sum over its n samples, the estimator of the diagnostics; not rsl_rl's analytic Gaussian KL,
                      which needs the old means the rollout does not keep); kl > 2 delta: lr = max(1e-5, lr / 1.5); 0 < kl < delta / 2:
                      lr = min(1e-2, lr * 1.5); otherwise (NaN and inf included) unchanged.  Each of the pair's two nets applies the
                      rule to its own lr with the pair's one kl.  The lr state is fp32 on the device (changes computed in fp64 and
                      rounded); it is loaded from the six Adam.lr at the start of each update and written back to them in the
                      synchronisation that ends it, so it carries over between updates and a value set between updates is honoured.
                      Turns the diagnostics on.  With target_kl the halt test comes first (a halted step changes no weight and no
                      lr); with max_grad_norm the gradient is clipped, then the step takes the adapted lr.  One launch per step
                      (mhppo_adam2_sched).  train_model_c / _d called outside update() take the plain path with Adam.lr.
  update() leaves the lr of every step (fp32 values; NaN for a step the target-KL halt skipped in "adaptive" mode) in `last_lrs`,
  train() appends each pair's lrs after the update to `ep_lrs`.  Checkpoints keep no lr: a resumed "adaptive" run restarts from
  the constructor's values.
Reward normalisation, also off by default (DESIGN.md §4 "Reward normalisation", §5 "Reward normalisation"):
  normalize_reward=False  True: SB3's VecNormalize reward path, each (car, env) column one env.  Once per rollout, at the start of
                      update(), the batch moments of two streams -- the forward running return g_t = gamma * g_{t-1} + r_t of the `rew`
                      buffer (cross / wait nets) and the episodic choice reward `rew_d` -- over the present columns (route >= 0) are
                      all-reduced and merged into the running state `reward_rms` (device fp64 [2][3], rows continuous / choice,
                      columns count / mean / var, starting at (1e-4, 0, 1)); every update then regresses on
                      r~ = clip(r / sqrt(var + 1e-8), -c, c) (fp64, rounded to fp32 once; no mean subtracted) in place of the raw
                      rewards: reward-to-go / GAE from r~, and r~_d as the choice critic's target and in its advantage.  A second
                      update() on the same rollout rescales with the current state and does not merge again; a state set between
                      updates is honoured.  The raw `rew`, `rl`, `rew_d` keep their values, so ep_reward_* stay raw.  update() leaves
                      `last_reward_norm` = {"continuous", "choice"} -> dict(count, mean, var, scale), train() appends it to
                      `ep_reward_norm`.  Checkpoints keep no statistics: a resumed run restarts them.
  clip_reward=None    c > 0 (+inf: no clipping) with normalize_reward=True; None means 10.0 (SB3's default).

One iteration = one 80-step episode in every env of the vectorised env.  Multi-GPU: one process per GPU, envs
sharded per rank; the only collectives are the all-reduce of the three advantage statistics and of the flat
gradient buffers (NCCL through torch.distributed), so an R-rank run performs the same update as one rank
holding all envs (SURVEY.md 8e).
"""
import ctypes as C
import math
import numbers
import os

import numpy as np
import torch

from . import _lib
from ._lib import check
from .policy import Adam, Model_PPO
from .rollout import Env_rollout


_USE_DIST = True
MAX_MINIBATCHES = 1024       # mhppo_minibatch_plan: 5 x B histogram bins per tile in shared memory
PAIRS = ("cross", "wait", "choice")
DIAG_ROW = 10                # fp64 record row of one step (include/mhppo.h, mhppo_ppo_grad_diag)
DIAG_FIELDS = [("epoch", np.int32), ("minibatch", np.int32), ("n", np.int64), ("actor_loss", np.float64), ("critic_loss", np.float64),
               ("approx_kl", np.float64), ("clip_fraction", np.float64), ("entropy", np.float64), ("explained_variance", np.float64),
               ("taken", np.bool_)]
GRAD_NORM_FIELDS = [("epoch", np.int32), ("minibatch", np.int32), ("actor_grad_norm", np.float64), ("critic_grad_norm", np.float64)]
LR_FIELDS = [("epoch", np.int32), ("minibatch", np.int32), ("actor_lr", np.float64), ("critic_lr", np.float64)]
LR_SCHEDULES = ("linear", "adaptive")
REWARD_STREAMS = ("continuous", "choice")
REWARD_RMS0 = ((1e-4, 0.0, 1.0), (1e-4, 0.0, 1.0))        # (count, mean, var) of each stream: SB3's RunningMeanStd(epsilon=1e-4)


def diag_ratios(sums, n, choice):
    """The diagnostics of one step from its record sums over all ranks (row layout of mhppo_ppo_grad_diag) and its sample count n:
    approx_kl = mean k3, clip_fraction, entropy (choice pair only, NaN otherwise: the Gaussian heads have a fixed variance) and the
    explained variance 1 - Var(R - V) / Var(R) with population variances, NaN when Var(R) = 0."""
    sums = [float(v) for v in sums]
    var_d = sums[6] / n - (sums[5] / n) ** 2
    var_r = sums[8] / n - (sums[7] / n) ** 2
    return dict(actor_loss=sums[0], critic_loss=sums[1], approx_kl=sums[2] / n, clip_fraction=sums[3] / n,
                entropy=sums[4] / n if choice else float("nan"), explained_variance=1.0 - var_d / var_r if var_r > 0 else float("nan"))


def _to_host_async(t):
    """An asynchronous device-to-host copy of t into pinned memory; returns (host tensor, event of the copy)."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    done = torch.cuda.Event()
    done.record(torch.cuda.current_stream(t.device))
    return host, done


def set_distributed(on):
    """Tests only: run a single-rank reference pass inside an initialised process group."""
    global _USE_DIST
    _USE_DIST = bool(on)


def _dist():
    import torch.distributed as dist
    return dist if (_USE_DIST and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) else None


def combine_stats(stats3):
    """(sum A, sum A^2, n) -> (mean, 1/(unbiased std + 1e-10), n): advantage normalisation of PY:787 from partial sums."""
    sA, sAA, n = float(stats3[0]), float(stats3[1]), float(stats3[2])
    if n < 1:
        return 0.0, 0.0, 0.0
    mean = sA / n
    var = max(sAA - n * mean * mean, 0.0) / (n - 1) if n > 1 else float("nan")
    std = math.sqrt(var) if n > 1 else float("nan")
    return mean, 1.0 / (std + 1e-10), n


def allreduce_sum_(t):
    d = _dist()
    if d is not None:
        d.all_reduce(t, op=d.ReduceOp.SUM)
    return t


class Algo_PPO:
    def __init__(self, policy_class, env, **hyperparameters):
        self._init_hyperparameters(hyperparameters)
        self._check_options()
        self.env = env
        self.max_steps = env.max_episode
        dev = env.device
        nc = 2 * env.nb_lines
        mk = lambda *a, **k: policy_class(*a, device=dev, **k)
        self.actor_net_cross = mk(self.num_states_c, self.num_actions, 1, nb_car=nc, mean=self.mean, std=self.std)      # PY:711-718
        self.actor_net_wait = mk(self.num_states_c, self.num_actions, 1, nb_car=nc, mean=self.mean, std=self.std)
        self.actor_net_choice = mk(self.num_states_d, 2, 2)
        self.critic_net_cross = mk(self.num_states_c, 1, 0)
        self.critic_net_wait = mk(self.num_states_c, 1, 0)
        self.critic_net_choice = mk(self.num_states_d, 1, 0)
        self.optimizer_critic_cross = Adam(self.critic_net_cross, self.critic_lr)                                        # PY:719-724
        self.optimizer_critic_wait = Adam(self.critic_net_wait, self.critic_lr)
        self.optimizer_critic_choice = Adam(self.critic_net_choice, self.critic_d_lr)
        self.optimizer_actor_cross = Adam(self.actor_net_cross, self.actor_lr)
        self.optimizer_actor_wait = Adam(self.actor_net_wait, self.actor_lr)
        self.optimizer_actor_choice = Adam(self.actor_net_choice, self.actor_d_lr)
        if not hasattr(self, "value_std"):
            self.value_std = 0.5                                                                                         # PY:726
        self.value_std_d = 0.1                                                                                           # PY:727 (unused by the reference's Categorical)
        self.rollout = Env_rollout(env, env.n_slots, self.max_steps, self.dt)
        if self.num_states_d != self.rollout.shape_env_d:
            raise ValueError("num_states_d = %s, but the choice features of this env have %d columns" % (self.num_states_d, self.rollout.shape_env_d))
        self.rollout.value_std = self.value_std
        self.ep_reward_cross, self.ep_reward_wait, self.ep_reward_choice, self.ep_scenario_balance = [], [], [], []
        L = _lib.lib()
        nbytes = max(L.mhppo_update_workspace_bytes(self.num_states_c), L.mhppo_update_workspace_bytes(self.num_states_d))
        self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        self._stats = torch.zeros(3, dtype=torch.float64, device=dev)
        self._diag = bool(self.diagnostics) or self.target_kl is not None or self.lr_schedule == "adaptive"
        self._steps = None                                # per pair, the steps of the update in progress (diagnostics, clipping)
        self._rec = None                                  # the record of the update in progress (diagnostics)
        self._norms = None                                # its gradient norms, fp64 [step][actor, critic] (clipping)
        self._halt = torch.zeros(3, dtype=torch.int32, device=dev)
        self.last_update_stats, self.ep_diagnostics = {}, []
        self.last_grad_norms, self.ep_grad_norms = {}, []
        self._lr0 = [(oa.lr, oc.lr) for _, (oa, oc) in self._pair_optimizers()]          # the constructor's lrs ("linear")
        self._lrs = None                                  # the lrs of the update in progress, fp64 [step][actor, critic] ("adaptive")
        if self.lr_schedule == "adaptive":               # the lr state, fp32 [pair][actor, critic], and its pinned staging copy
            self._lr_dev = torch.zeros(len(PAIRS), 2, dtype=torch.float32, device=dev)
            self._lr_host = torch.zeros(len(PAIRS), 2, dtype=torch.float32, pin_memory=True)
        self.last_lrs, self.ep_lrs = {}, []
        self.reward_rms = self._rn_moments = None            # reward normalisation: running state and this rollout's batch moments
        if self.normalize_reward:
            self.reward_rms = torch.tensor(REWARD_RMS0, dtype=torch.float64, device=dev)
            self._rn_moments = torch.zeros(6, dtype=torch.float64, device=dev)
        self._rn_iteration = None                            # the rollout whose batch reward_rms last merged
        self.last_reward_norm, self.ep_reward_norm = {}, []
        self._loss = torch.zeros(2, dtype=torch.float64, device=dev)
        self.last_losses = {}
        self._sel_cache = {}
        self._mb = {}                                    # minibatch plan buffers (n_minibatches mode)
        # one contiguous gradient buffer per (actor, critic) pair: a single all-reduce per epoch carries both (with diagnostics also
        # the actor's k3 sum in one more fp32 slot, which the target-KL halt reads)
        self._gbuf, self._klslot = {}, {}
        for name, actor, critic in (("cross", self.actor_net_cross, self.critic_net_cross), ("wait", self.actor_net_wait, self.critic_net_wait),
                                    ("choice", self.actor_net_choice, self.critic_net_choice)):
            np_ = actor.n_param + critic.n_param
            g = torch.zeros(np_ + (1 if self._diag else 0), device=dev)
            actor.grad, critic.grad = g[:actor.n_param], g[actor.n_param:np_]
            self._gbuf[id(actor)] = g
            self._klslot[id(actor)] = g[np_:]
        self.sync_parameters()

    def sync_parameters(self):
        """Multi-GPU: every rank must hold rank 0's parameters and optimiser state (only gradients and advantage statistics
        are all-reduced afterwards, so the replicas then stay identical).  Called after construction and loading()."""
        d = _dist()
        if d is None:
            return
        for _, _, net in self._nets():
            for t in (net.flat, net.m, net.v):
                d.broadcast(t, src=0)
            step = torch.tensor([net.step], dtype=torch.int64, device=net.flat.device)
            d.broadcast(step, src=0)
            net.step = int(step.item())

    def _init_hyperparameters(self, hyperparameters):
        """PY:919-933."""
        self.num_algo, self.total_loop, self.batch_size, self.gamma = 1, 0, 2048, 0.99
        self.critic_lr, self.actor_lr, self.critic_d_lr, self.actor_d_lr = 1e-3, 3e-4, 1e-3, 3e-4
        self.num_states_c, self.num_states_d, self.num_actions, self.mean, self.std, self.dt = 13, None, 1, -1.0, 3.0, 0.3
        self.gae_lambda, self.entropy_coef = None, 0.0                     # options beyond the reference (module docstring)
        self.n_minibatches = None
        self.diagnostics, self.target_kl = False, None
        self.max_grad_norm = None
        self.lr_schedule, self.desired_kl, self.lr_anneal_iterations = None, None, None
        self.normalize_reward, self.clip_reward = False, None
        for k, v in hyperparameters.items():
            setattr(self, k, v)

    def _check_options(self):
        real = lambda v: isinstance(v, numbers.Real) and not isinstance(v, bool)
        lam, c = self.gae_lambda, self.entropy_coef
        if lam is not None:
            if not (real(lam) and 0.0 <= float(lam) <= 1.0):
                raise ValueError("gae_lambda must be None or a number in [0, 1], got %r" % (lam,))
            if not (real(self.gamma) and 0.0 <= float(self.gamma) <= 1.0):
                raise ValueError("GAE needs gamma in [0, 1], got %r" % (self.gamma,))
        if not (real(c) and math.isfinite(float(c)) and float(c) >= 0.0):
            raise ValueError("entropy_coef must be a finite number >= 0, got %r" % (c,))
        B = self.n_minibatches
        if B is not None and not (isinstance(B, numbers.Integral) and not isinstance(B, bool) and 1 <= int(B) <= MAX_MINIBATCHES):
            raise ValueError("n_minibatches must be None or an integer in [1, %d], got %r" % (MAX_MINIBATCHES, B))
        if not isinstance(self.diagnostics, bool):
            raise ValueError("diagnostics must be a bool, got %r" % (self.diagnostics,))
        d = self.target_kl
        if d is not None and not (real(d) and math.isfinite(float(d)) and float(d) > 0.0):
            raise ValueError("target_kl must be None or a finite number > 0, got %r" % (d,))
        g = self.max_grad_norm
        if g is not None and not (real(g) and float(g) > 0.0):
            raise ValueError("max_grad_norm must be None or a number > 0 (inf: record the norms, never clip), got %r" % (g,))
        s, d, K = self.lr_schedule, self.desired_kl, self.lr_anneal_iterations
        if not (s is None or (isinstance(s, str) and s in LR_SCHEDULES)):
            raise ValueError("lr_schedule must be None, 'linear' or 'adaptive', got %r" % (s,))
        if s == "adaptive":
            if not (real(d) and math.isfinite(float(d)) and float(d) > 0.0):
                raise ValueError("lr_schedule='adaptive' needs desired_kl, a finite number > 0, got %r" % (d,))
        elif d is not None:
            raise ValueError("desired_kl is an option of lr_schedule='adaptive', got %r with lr_schedule=%r" % (d, s))
        if s == "linear":
            if not (isinstance(K, numbers.Integral) and not isinstance(K, bool) and int(K) >= 1):
                raise ValueError("lr_schedule='linear' needs lr_anneal_iterations, an integer >= 1, got %r" % (K,))
        elif K is not None:
            raise ValueError("lr_anneal_iterations is an option of lr_schedule='linear', got %r with lr_schedule=%r" % (K, s))
        if not isinstance(self.normalize_reward, bool):
            raise ValueError("normalize_reward must be a bool, got %r" % (self.normalize_reward,))
        c = self.clip_reward
        if c is not None:
            if not self.normalize_reward:
                raise ValueError("clip_reward is an option of normalize_reward=True, got %r with normalize_reward=False" % (c,))
            if not (real(c) and float(c) > 0.0):
                raise ValueError("clip_reward must be None or a number > 0 (inf: no clipping), got %r" % (c,))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    # -- one epoch of train_model_c (PY:778-815) on the cross (want=0) or wait (want=1) buffer ------------------
    def _selection(self, want):
        """Compacted (car, env) columns routed to the cross (0) / wait (1) buffer, or the existing cars (want=None)."""
        r = self.rollout
        key = (r.iteration, r.route.data_ptr(), int(r.route._version), int(r.exist._version))
        if self._sel_cache.get("key") != key:
            self._sel_cache = {"key": key}
        if want not in self._sel_cache:
            mask = (r.exist.view(-1) != 0) if want is None else (r.route.view(-1) == want)
            sel = torch.nonzero(mask).view(-1).to(torch.int32)
            self._sel_cache[want] = (sel if sel.numel() else torch.zeros(1, dtype=torch.int32, device=mask.device), sel.numel())
        return self._sel_cache[want]

    def _global_count(self, want, local):
        """Samples of this buffer over all ranks (the denominators of the losses, PY:806-809); the selection is fixed for
        the 10 epochs of an update, so the all-reduce happens once per buffer."""
        k = ("n", want)
        if k not in self._sel_cache:
            t = torch.tensor([float(local)], dtype=torch.float64, device=self.rollout.route.device)
            self._sel_cache[k] = int(allreduce_sum_(t).item())
        return self._sel_cache[k]

    def train_model_c(self, actor, critic, opti_actor, opti_critic, want):
        r = self.rollout
        idx, K = self._selection(want)                                      # K == 0 still runs (zero partials): other ranks may have samples
        n = self._global_count(want, K * (r.S // r.M))             # sample slots: S = T * M, M = C * N columns
        if n < 1:
            return False                                     # PY:869/874: the net is skipped when its buffer is empty
        self._epoch_c(actor, critic, opti_actor, opti_critic, want, idx.data_ptr(), K, n)
        return True

    def _epoch_c(self, actor, critic, opti_actor, opti_critic, want, idx, K, n):
        """One gradient step of the pair on the K local columns of the int32 list at device address `idx`; n = the sample
        count over all ranks (the whole buffer, or one minibatch of it)."""
        r, L, st = self.rollout, _lib.lib(), self._stream()
        ws = self._ws.data_ptr()
        row = self._diag_row(want, n)
        if self.gae_lambda is not None:
            # GAE: fixed targets ret and advantages ret - V_old of this update; the critic pass must not overwrite V_old
            stats = self._gae_stats()
            if row is not None:
                check(L.mhppo_critic_grad_diag(13, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, critic.flat.data_ptr(), r.ret.data_ptr(), 1.0 / n,
                                               critic.grad.data_ptr(), self._loss.data_ptr() + 8, None, None, row, ws, st))
                self._actor_diag(1, r.obs_c, 13, r.S, idx, K, actor, r.act, r.logp, r.ret, r.V, stats.data_ptr() + 24 * want, n, 0.0, 0.0, 0.0, row)
            else:
                check(L.mhppo_ppo_grad(13, 0, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, critic.flat.data_ptr(), None, None,
                                       r.ret.data_ptr(), None, 0.0, 0.0, 1.0 / n, 0.0, 0.0, critic.grad.data_ptr(), self._loss.data_ptr() + 8,
                                       ws, st))
                check(L.mhppo_ppo_grad_dev(13, 1, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, actor.flat.data_ptr(),
                                           r.act.data_ptr(), r.logp.data_ptr(), r.ret.data_ptr(), r.V.data_ptr(), stats.data_ptr() + 24 * want,
                                           1.0 / n, 0.0, 0.0, actor.grad.data_ptr(), self._loss.data_ptr(), ws, st))
            self._step_pair(actor, critic, opti_actor, opti_critic, n, row)
            return
        # critic pass first: its forward is V = critic(s) of PY:785, so the same kernel returns V and the advantage statistics
        if row is not None:
            check(L.mhppo_critic_grad_diag(13, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, critic.flat.data_ptr(), r.rtg.data_ptr(), 1.0 / n,
                                           critic.grad.data_ptr(), self._loss.data_ptr() + 8, r.V.data_ptr(), self._stats.data_ptr(), row, ws, st))
        else:
            check(L.mhppo_critic_grad_stats(13, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, critic.flat.data_ptr(),
                                            r.rtg.data_ptr(), 1.0 / n, critic.grad.data_ptr(), self._loss.data_ptr() + 8,
                                            r.V.data_ptr(), self._stats.data_ptr(), ws, st))
        allreduce_sum_(self._stats)                          # (sum A, sum A^2, n) over all ranks; normalised inside the actor kernel
        if row is not None:
            self._actor_diag(1, r.obs_c, 13, r.S, idx, K, actor, r.act, r.logp, r.rtg, r.V, self._stats.data_ptr(), n, 0.0, 0.0, 0.0, row)
        else:
            check(L.mhppo_ppo_grad_dev(13, 1, r.obs_c.data_ptr(), 13, r.S, idx, K, r.M, actor.flat.data_ptr(),
                                       r.act.data_ptr(), r.logp.data_ptr(), r.rtg.data_ptr(), r.V.data_ptr(), self._stats.data_ptr(), 1.0 / n,
                                       0.0, 0.0, actor.grad.data_ptr(), self._loss.data_ptr(), ws, st))
        self._step_pair(actor, critic, opti_actor, opti_critic, n, row)

    def _actor_diag(self, head, x, D, S, idx, K, actor, act, logp, rtg, V, stats_ptr, n, f0, f1, c, row):
        """The actor pass with diagnostics: record row `row` (device address) and the k3 sum into the pair's extra gradient slot."""
        r = self.rollout
        check(_lib.lib().mhppo_ppo_grad_diag(D, head, x.data_ptr(), D, S, idx, K, r.M, actor.flat.data_ptr(), act.data_ptr(), logp.data_ptr(),
                                             rtg.data_ptr(), V.data_ptr(), stats_ptr, 1.0 / n, f0, f1, c, actor.grad.data_ptr(),
                                             self._loss.data_ptr(), self._klslot[id(actor)].data_ptr(), row, self._ws.data_ptr(),
                                             self._stream()))

    def _prepare_gae(self):
        """GAE mode, once per update before the epochs: V_old of both critics, the returns and the advantage statistics of
        the cross and wait samples, all-reduced over the ranks once."""
        r = self.rollout
        _, stats6 = r.gae(self.critic_net_cross, self.critic_net_wait, self.gamma, self.gae_lambda,
                          selections=(self._selection(0), self._selection(1)), workspace=self._ws,
                          rew=r.rew_n if self.normalize_reward else None)
        self._sel_cache["gae"] = allreduce_sum_(stats6)

    def _normalize_rewards(self):
        """Reward normalisation, once per update after the raw mhppo_returns (which forms rew_d): this rollout's batch moments of
        both streams, all-reduced over the ranks (one device tensor, no host synchronisation), merged into reward_rms on the device
        unless this rollout's batch is in it already; then r~ into rollout.rew_n / rew_dn and the reward-to-go from r~ (GAE mode
        forms its returns from rew_n in _prepare_gae).  Returns the asynchronous host copy of reward_rms (host tensor, event)."""
        r, L, st = self.rollout, _lib.lib(), self._stream()
        rms = self.reward_rms
        if not (isinstance(rms, torch.Tensor) and rms.dtype == torch.float64 and rms.shape == (2, 3) and rms.device == self._stats.device
                and rms.is_contiguous()):
            raise ValueError("reward_rms must be a contiguous float64 tensor of shape (2, 3) on %s" % (self._stats.device,))
        if r.rew_n is None:
            r.rew_n, r.rew_dn = torch.zeros_like(r.rew), torch.zeros_like(r.rew_d)
        check(L.mhppo_reward_moments(r.rew.data_ptr(), r.rew_d.data_ptr(), r.route.data_ptr(), r.T, r.M, float(self.gamma),
                                     self._rn_moments.data_ptr(), self._ws.data_ptr(), st))
        allreduce_sum_(self._rn_moments)
        merge = r.iteration != self._rn_iteration
        self._rn_iteration = r.iteration
        clip = 10.0 if self.clip_reward is None else float(self.clip_reward)
        check(L.mhppo_reward_normalize(r.rew.data_ptr(), r.rew_d.data_ptr(), r.T, r.M, self._rn_moments.data_ptr(), rms.data_ptr(),
                                       int(merge), clip, r.rew_n.data_ptr(), r.rew_dn.data_ptr(), st))
        if self.gae_lambda is None:
            r.futur_rewards(r.rew_n)
        return _to_host_async(rms)

    def _gae_stats(self):
        if "gae" not in self._sel_cache:                    # train_model_c called outside update() on a new rollout
            self._prepare_gae()
        return self._sel_cache["gae"]

    def _step_pair(self, actor, critic, opti_actor, opti_critic, n=None, row=None):
        """All-reduce the pair's packed gradients (one collective) and take both Adam steps in one launch (PY:810-815); with
        target_kl, the launch that halts the pair on the device (its step counts are settled after the update, _diag_finish); with
        max_grad_norm, the launch that clips each net's gradient first (inside update() it also records the two norms); inside an
        update with lr_schedule="adaptive", the launch that first adapts the pair's two lrs on the device (mhppo_adam2_sched)."""
        allreduce_sum_(self._gbuf[id(actor)])
        actor.step += 1; critic.step += 1
        L = _lib.lib()
        adam = (actor.flat.data_ptr(), actor.grad.data_ptr(), actor.m.data_ptr(), actor.v.data_ptr(), actor.n_param, opti_actor.lr, actor.step,
                critic.flat.data_ptr(), critic.grad.data_ptr(), critic.m.data_ptr(), critic.v.data_ptr(), critic.n_param, opti_critic.lr,
                critic.step, 0.9, 0.999, 1e-8)
        halt = None
        if row is not None and self.target_kl is not None:
            halt = (self._klslot[id(actor)].data_ptr(), 1.5 * float(self.target_kl) * n, self._halt.data_ptr() + 4 * self._rec_pair, row)
        norms = None if self._norms is None else self._norms.data_ptr() + 16 * self._rec_i
        if self._lrs is not None:
            g = math.inf if self.max_grad_norm is None else float(self.max_grad_norm)
            check(L.mhppo_adam2_sched(*adam, g, norms, *(halt or (None, 0.0, None, None)), self._lr_dev.data_ptr() + 8 * self._rec_pair,
                                      self._klslot[id(actor)].data_ptr(), float(n), float(self.desired_kl),
                                      self._lrs.data_ptr() + 16 * self._rec_i, self._stream()))
        elif self.max_grad_norm is not None:
            check(L.mhppo_adam2_clip(*adam, float(self.max_grad_norm), norms, *(halt or (None, 0.0, None, None)), self._stream()))
        elif halt is not None:
            check(L.mhppo_adam2_halt(*adam, *halt, self._stream()))
        else:
            check(L.mhppo_adam2(*adam, self._stream()))

    # -- one epoch of train_model_d (PY:818-851) on the choice buffer -------------------------------------------
    def train_model_d(self, actor, critic, opti_actor, opti_critic):
        idx, K = self._selection(None)
        n = self._global_count(None, K)
        if n < 1:
            return False
        self._epoch_d(actor, critic, opti_actor, opti_critic, idx.data_ptr(), K, n, lambda: self._action_fractions(n))
        return True

    def _epoch_d(self, actor, critic, opti_actor, opti_critic, idx, K, n, fractions):
        """One gradient step of the choice pair on the K local columns at device address `idx`; n = the sample count over all
        ranks, fractions() = (f0, f1) of those n samples."""
        r, L, st = self.rollout, _lib.lib(), self._stream()
        ws, D = self._ws.data_ptr(), r.shape_env_d
        rew_d = r.rew_dn if self.normalize_reward else r.rew_d       # the choice target: normalised (reward normalisation) or raw
        row = self._diag_row(2, n)
        if row is not None:
            check(L.mhppo_critic_grad_diag(D, r.obs_d.data_ptr(), D, r.M, idx, K, r.M, critic.flat.data_ptr(), rew_d.data_ptr(), 1.0 / n,
                                           critic.grad.data_ptr(), self._loss.data_ptr() + 8, r.V_d.data_ptr(), self._stats.data_ptr(), row, ws, st))
        else:
            check(L.mhppo_critic_grad_stats(D, r.obs_d.data_ptr(), D, r.M, idx, K, r.M, critic.flat.data_ptr(),
                                            rew_d.data_ptr(), 1.0 / n, critic.grad.data_ptr(), self._loss.data_ptr() + 8,
                                            r.V_d.data_ptr(), self._stats.data_ptr(), ws, st))
        allreduce_sum_(self._stats)
        f0, f1 = fractions()
        if row is not None:
            self._actor_diag(2, r.obs_d, D, r.M, idx, K, actor, r.act_d, r.logp_d, rew_d, r.V_d, self._stats.data_ptr(), n, f0, f1,
                             float(self.entropy_coef), row)
            self._step_pair(actor, critic, opti_actor, opti_critic, n, row)
            return
        if self.entropy_coef:
            check(L.mhppo_ppo_grad_ent(D, 2, r.obs_d.data_ptr(), D, r.M, idx, K, r.M, actor.flat.data_ptr(),
                                       r.act_d.data_ptr(), r.logp_d.data_ptr(), rew_d.data_ptr(), r.V_d.data_ptr(), self._stats.data_ptr(),
                                       1.0 / n, f0, f1, float(self.entropy_coef), actor.grad.data_ptr(), self._loss.data_ptr(), ws, st))
            self._step_pair(actor, critic, opti_actor, opti_critic)
            return
        check(L.mhppo_ppo_grad_dev(D, 2, r.obs_d.data_ptr(), D, r.M, idx, K, r.M, actor.flat.data_ptr(),
                                   r.act_d.data_ptr(), r.logp_d.data_ptr(), rew_d.data_ptr(), r.V_d.data_ptr(), self._stats.data_ptr(),
                                   1.0 / n, f0, f1, actor.grad.data_ptr(), self._loss.data_ptr(), ws, st))
        self._step_pair(actor, critic, opti_actor, opti_critic)

    def _action_fractions(self, n):
        """Fractions of the choice samples (all ranks) whose action is 0 / 1: the (M, M) broadcast of PY:834-842 collapses to
        them.  Fixed for the epochs of an update: counted once per rollout."""
        if "f01" not in self._sel_cache:
            r = self.rollout
            ex = r.exist.view(-1) != 0
            cnt = torch.stack([(ex & (r.act_d == 0)).sum(), (ex & (r.act_d == 1)).sum()]).double()
            cnt = allreduce_sum_(cnt).cpu()
            self._sel_cache["f01"] = (float(cnt[0]) / n, float(cnt[1]) / n)
        return self._sel_cache["f01"]

    def update(self, epochs=10):
        """The update half of train() (PY:866-882): 10 x (cross, wait) then 10 x choice; with n_minibatches = B, B steps per net
        and epoch (_update_minibatches)."""
        self.rollout.value_std = self.value_std
        self.rollout._set_head(self.actor_net_cross)
        self.rollout.futur_rewards()                    # also the choice reward rew_d, which GAE mode uses too
        pending_rn = self._normalize_rewards() if self.normalize_reward else None
        if self.gae_lambda is not None:
            self._prepare_gae()
        clip, sched = self.max_grad_norm is not None, self.lr_schedule
        if sched == "linear":
            frac = max(0.0, 1.0 - self.total_loop / int(self.lr_anneal_iterations))
            for (_, (oa, oc)), (la, lc) in zip(self._pair_optimizers(), self._lr0):
                oa.lr, oc.lr = la * frac, lc * frac
        if self._diag or clip or sched is not None:
            self._steps_begin(epochs, clip)
        try:
            if self.n_minibatches is not None:
                self._update_minibatches(epochs)
            else:
                for e in range(epochs):
                    self._pos = (e, 0)
                    self.train_model_c(self.actor_net_cross, self.critic_net_cross, self.optimizer_actor_cross, self.optimizer_critic_cross, 0)
                    self.train_model_c(self.actor_net_wait, self.critic_net_wait, self.optimizer_actor_wait, self.optimizer_critic_wait, 1)
                for e in range(epochs):
                    self._pos = (e, 0)
                    self.train_model_d(self.actor_net_choice, self.critic_net_choice, self.optimizer_actor_choice, self.optimizer_critic_choice)
            pending = self._diag_fetch() if self._diag else None
            pending_norms = _to_host_async(self._norms[:self._n_steps]) if clip else None
            pending_lrs = (_to_host_async(self._lrs[:self._n_steps]), _to_host_async(self._lr_dev)) if self._lrs is not None else None
        finally:
            self._steps_done, self._steps = self._steps, None
            self._rec = self._norms = self._lrs = None   # train_model_c / _d outside update() take the plain path
        failed = _lib.lib().mhppo_tc_failures()          # (synchronises the device: the copies have landed with it)
        if pending is not None:
            host, done = pending
            done.synchronize()
            self._diag_finish(host.numpy())              # step counts settled even when the update is reported broken below
        if pending_norms is not None:
            host, done = pending_norms
            done.synchronize()
            self._grad_norms_finish(host.numpy())
        if pending_rn is not None:
            host, done = pending_rn
            done.synchronize()
            self.last_reward_norm = {k: dict(count=c, mean=m, var=v, scale=math.sqrt(v + 1e-8))
                                     for k, (c, m, v) in zip(REWARD_STREAMS, host.tolist())}
        if pending_lrs is not None:
            for _, done in pending_lrs:
                done.synchronize()
            self._lrs_finish(pending_lrs[0][0].numpy(), pending_lrs[1][0].numpy())
        elif sched == "linear":
            self._lrs_finish(None, None)
        if failed:                                       # a tensor-core kernel gave up waiting for its MMAs: its gradients are garbage
            raise RuntimeError("a tcgen05 kernel of the update timed out on its mbarrier; the parameters of this update are not "
                               "trustworthy (reload a checkpoint; MHPPO_MLP=ffma selects the CUDA-core kernels)")

    # -- per-step records of an update: diagnostics (diagnostics=True / target_kl) and gradient norms (max_grad_norm) ----------
    def _steps_begin(self, epochs, clip):
        """The step bookkeeping of this update; with diagnostics a zeroed record of one fp64 row per possible step and the pairs'
        halt flags cleared, with clipping one fp64 (actor, critic) norm row per possible step.  Both are indexed by the same step
        counter, so their rows line up."""
        B = int(self.n_minibatches) if self.n_minibatches is not None else 1
        dev = self._stats.device
        self._steps = {p: [] for p in PAIRS}             # per pair: (epoch, minibatch, n, step index), in launch order
        self._n_steps = 0
        self._pos = (0, 0)
        if self._diag:
            self._rec = torch.zeros(3 * epochs * B, DIAG_ROW, dtype=torch.float64, device=dev)
            self._rec_steps0 = {p: (a.step, c.step) for p, a, c in self._pair_nets()}
            if self.target_kl is not None:
                self._halt.zero_()
        if clip:
            self._norms = torch.zeros(3 * epochs * B, 2, dtype=torch.float64, device=dev)
        if self.lr_schedule == "adaptive":
            # the lr state from the six Adam.lr (the previous update's synchronisation has ended every use of the staging copy)
            self._lr_host.copy_(torch.tensor([[oa.lr, oc.lr] for _, (oa, oc) in self._pair_optimizers()], dtype=torch.float32))
            self._lr_dev.copy_(self._lr_host, non_blocking=True)
            self._lrs = torch.full((3 * epochs * B, 2), math.nan, dtype=torch.float64, device=dev)

    def _pair_optimizers(self):
        return (("cross", (self.optimizer_actor_cross, self.optimizer_critic_cross)), ("wait", (self.optimizer_actor_wait, self.optimizer_critic_wait)),
                ("choice", (self.optimizer_actor_choice, self.optimizer_critic_choice)))

    def _pair_nets(self):
        return (("cross", self.actor_net_cross, self.critic_net_cross), ("wait", self.actor_net_wait, self.critic_net_wait),
                ("choice", self.actor_net_choice, self.critic_net_choice))

    def _diag_row(self, pair, n):
        """Counts a step of pair 0 / 1 / 2 with n samples over all ranks (inside update(), with diagnostics or clipping) and returns
        the device address of its record row; None outside update() or without diagnostics."""
        if self._steps is None:
            return None
        i = self._n_steps
        self._n_steps += 1
        self._steps[PAIRS[pair]].append((self._pos[0], self._pos[1], int(n), i))
        self._rec_pair, self._rec_i = pair, i
        return None if self._rec is None else self._rec.data_ptr() + 8 * DIAG_ROW * i

    def _diag_fetch(self):
        """One all-reduce of the record's sums over the ranks (the taken flags are the same on every rank) and one asynchronous
        device-to-host copy of the used rows into pinned memory; returns (host tensor, event of the copy).  The host waits for it
        in the same synchronisation as the mhppo_tc_failures copy that ends every update."""
        used = self._n_steps
        if _dist() is not None and used:
            s = self._rec[:used, :DIAG_ROW - 1].contiguous()
            allreduce_sum_(s)
            self._rec[:used, :DIAG_ROW - 1] = s
        return _to_host_async(self._rec[:used])

    def _diag_finish(self, host):
        """last_update_stats from the copied record; with target_kl, each pair's Adam step counts become the steps it took."""
        out = {}
        for p, actor, critic in self._pair_nets():
            steps = self._steps_done[p]
            a = np.zeros(len(steps), dtype=DIAG_FIELDS)
            for j, (e, b, n, i) in enumerate(steps):
                a[j]["epoch"], a[j]["minibatch"], a[j]["n"] = e, b, n
                for k, v in diag_ratios(host[i, :DIAG_ROW - 1], n, p == "choice").items():
                    a[j][k] = v
                a[j]["taken"] = bool(host[i, DIAG_ROW - 1]) if self.target_kl is not None else True
            out[p] = a
            if self.target_kl is not None:
                s0a, s0c = self._rec_steps0[p]
                actor.step, critic.step = s0a + int(a["taken"].sum()), s0c + int(a["taken"].sum())
        self.last_update_stats = out

    def _grad_norms_finish(self, host):
        """last_grad_norms from the copied norms (the same on every rank: they are taken after the gradient all-reduce)."""
        out = {}
        for p in PAIRS:
            steps = self._steps_done[p]
            a = np.zeros(len(steps), dtype=GRAD_NORM_FIELDS)
            for j, (e, b, n, i) in enumerate(steps):
                a[j]["epoch"], a[j]["minibatch"] = e, b
                a[j]["actor_grad_norm"], a[j]["critic_grad_norm"] = host[i]
            out[p] = a
        self.last_grad_norms = out

    def _lrs_finish(self, rows, state):
        """last_lrs: per pair and launched step the (actor, critic) lr the step used, fp32 values.  "adaptive": rows = the copied
        per-step lrs (NaN where the target-KL halt skipped the step), state = the final device lr state, which the six Adam.lr take
        over; "linear" (both None): every step used the Adam.lr set at the start of the update."""
        if state is not None:
            for (_, (oa, oc)), (la, lc) in zip(self._pair_optimizers(), state.tolist()):
                oa.lr, oc.lr = la, lc
        out = {}
        for p, (oa, oc) in self._pair_optimizers():
            steps = self._steps_done[p]
            a = np.zeros(len(steps), dtype=LR_FIELDS)
            for j, (e, b, n, i) in enumerate(steps):
                a[j]["epoch"], a[j]["minibatch"] = e, b
                a[j]["actor_lr"], a[j]["critic_lr"] = rows[i] if rows is not None else (np.float32(oa.lr), np.float32(oc.lr))
            out[p] = a
        self.last_lrs = out

    def grad_norms_summary(self):
        """Per pair: the means of last_grad_norms' actor and critic norms over the launched steps, and the steps launched."""
        return {p: dict(actor_grad_norm=float(np.mean(a["actor_grad_norm"])) if len(a) else float("nan"),
                        critic_grad_norm=float(np.mean(a["critic_grad_norm"])) if len(a) else float("nan"), steps_launched=int(len(a)))
                for p, a in self.last_grad_norms.items()}

    def diagnostics_summary(self):
        """Per pair: the means of last_update_stats' float fields over the launched steps, and the steps launched / taken."""
        out = {}
        for p, a in self.last_update_stats.items():
            d = {k: (float(np.mean(a[k])) if len(a) else float("nan")) for k, t in DIAG_FIELDS if t is np.float64}
            d["steps_launched"], d["steps_taken"] = int(len(a)), int(a["taken"].sum())
            out[p] = d
        return out

    # -- minibatch mode (n_minibatches = B) ----------------------------------------------------------------------
    def minibatch_plan(self, epochs):
        """The plan of this update (mhppo_minibatch_plan on the last rollout): per epoch the bucket-major column lists of the
        cross, wait and existing-car selections.  Returns (local, global) int64 numpy arrays [epochs][5][B] of the bucket sizes
        (rows: cross, wait, existing, existing with choice action 0, with action 1), this rank's and all ranks' (one
        all-reduce); the lists stay in self._mb["lists"] ([epochs][3][M] int32).  One device-to-host copy."""
        r, B, dev = self.rollout, int(self.n_minibatches), self.rollout.route.device
        if self._mb.get("key") != (epochs, B, r.M):
            self._mb = dict(key=(epochs, B, r.M), lists=torch.empty(epochs * 3 * r.M, dtype=torch.int32, device=dev),
                            offsets=torch.empty(epochs * 3 * (B + 1), dtype=torch.int64, device=dev),
                            counts=torch.empty(2, epochs * 5 * B, dtype=torch.int64, device=dev),
                            ws=torch.empty(1280 * epochs * B, dtype=torch.uint8, device=dev))
        p = self._mb
        check(_lib.lib().mhppo_minibatch_plan(C.byref(r._cfg), r.route.data_ptr(), r.exist.data_ptr(), r.act_d.data_ptr(),
                                              (r.iteration - 1) & 0xFFFFFFFF, epochs, B, p["lists"].data_ptr(), p["offsets"].data_ptr(),
                                              p["counts"].data_ptr(), p["ws"].data_ptr(), self._stream()))
        p["counts"][1].copy_(p["counts"][0])
        allreduce_sum_(p["counts"][1])
        cnt = p["counts"].cpu().numpy().reshape(2, epochs, 5, B)
        return cnt[0], cnt[1]

    def _update_minibatches(self, epochs):
        """Per epoch: cross on buckets 0..B-1, then wait on buckets 0..B-1; then the choice epochs on the existing cars.  Each
        minibatch is one call of the epoch body on its slice of the plan's list, with n = its sample count over all ranks; one
        with n < 2 takes no step (its unbiased std would be NaN).  Every rank takes the same decisions from the global counts."""
        r, B = self.rollout, int(self.n_minibatches)
        loc, glob = self.minibatch_plan(epochs)
        base, T = self._mb["lists"].data_ptr(), r.S // r.M

        def slices(e, s):
            off = np.concatenate(([0], np.cumsum(loc[e, s])))
            for b in range(B):
                yield b, base + 4 * ((e * 3 + s) * r.M + int(off[b])), int(loc[e, s, b]), int(glob[e, s, b])
        pairs = ((0, self.actor_net_cross, self.critic_net_cross, self.optimizer_actor_cross, self.optimizer_critic_cross),
                 (1, self.actor_net_wait, self.critic_net_wait, self.optimizer_actor_wait, self.optimizer_critic_wait))
        for e in range(epochs):
            for want, actor, critic, oa, oc in pairs:
                for b, idx, K, g in slices(e, want):
                    self._pos = (e, b)
                    if T * g >= 2:
                        self._epoch_c(actor, critic, oa, oc, want, idx, K, T * g)
        for e in range(epochs):
            for b, idx, K, n in slices(e, 2):
                self._pos = (e, b)
                if n >= 2:          # f0, f1 as _action_fractions forms them (float(count) / n): B = 1 is the default path bit for bit
                    f01 = (float(glob[e, 3, b]) / n, float(glob[e, 4, b]) / n)
                    self._epoch_d(self.actor_net_choice, self.critic_net_choice, self.optimizer_actor_choice, self.optimizer_critic_choice,
                                  idx, K, n, lambda f01=f01: f01)

    # file-name stems of the three drivers: PY:908 / NB2 (coop) / NB1 (naif, "acc6")
    _STEM = {"coop_scalable": "pappo-scalable-coop", "coop": "pappo-coop", "naif": "pappo-acc6", "stop": "pappo-acc6"}
    _TRACE = "load_model/parameters/{stem}-{num_algo:02d}-{name}-step-{epoch:03d}000.npy"

    def train(self, nb_loop, verbose=False, root=".", save_traces=True):
        """Training loop (PY:854-917); ends by writing the four learning-curve traces with the reference's file names
        (PY:908-916) under `root`, so a run can be laid next to the reference's load_model/parameters/*.npy."""
        for ep in range(nb_loop):
            self.rollout.iterations_rand(self.actor_net_cross, self.actor_net_wait, self.actor_net_choice)
            self.update()
            cross, wait, choice, (nc, nw, nd) = self._global_rewards()
            if cross is not None:
                self.ep_reward_cross.append(float(cross))
            if wait is not None:
                self.ep_reward_wait.append(float(wait))
            self.ep_reward_choice.append(float(choice))
            self.ep_scenario_balance.append([nc, nw])
            if self._diag:
                self.ep_diagnostics.append(self.diagnostics_summary())
            if self.max_grad_norm is not None:
                self.ep_grad_norms.append(self.grad_norms_summary())
            if self.lr_schedule is not None:
                self.ep_lrs.append({p: dict(actor_lr=oa.lr, critic_lr=oc.lr) for p, (oa, oc) in self._pair_optimizers()})
            if self.normalize_reward:
                self.ep_reward_norm.append(self.last_reward_norm)
            self.total_loop += 1
            if verbose:
                print("Episode * {} * cross {:.4f} wait {:.4f} choice {:.4f}  (#cross {} #wait {})".format(
                    ep, np.mean(self.ep_reward_cross[-10:] or [0]), np.mean(self.ep_reward_wait[-10:] or [0]),
                    np.mean(self.ep_reward_choice[-10:]), nc, nw))
        d = _dist()
        if save_traces and (d is None or d.get_rank() == 0):
            for name, arr in (("reward_cross", np.array(self.ep_reward_cross)), ("reward_wait", np.array(self.ep_reward_wait)),
                              ("reward_choice", np.array(self.ep_reward_choice)),
                              ("scenario_balance", np.array(self.ep_scenario_balance).reshape((-1, 2)))):
                path = os.path.join(root, self._TRACE.format(stem=self._STEM[self.env.variant], num_algo=self.num_algo,
                                                             epoch=int(self.total_loop / 1000), name=name))
                os.makedirs(os.path.dirname(path), exist_ok=True)
                np.save(path, arr)

    def _global_rewards(self):
        """Mean immediate rewards per buffer and the sample counts (PY:885-906), over the envs of ALL ranks."""
        r = self.rollout
        rew = r.rew.view(r.T, r.C, r.N)
        mc, mw, ex = (r.route == 0), (r.route == 1), (r.exist != 0)
        t = torch.stack([rew[:, mc].sum().double(), mc.sum().double() * r.T, rew[:, mw].sum().double(), mw.sum().double() * r.T,
                         r.rew_d.view(r.C, r.N)[ex].sum().double(), ex.sum().double()])
        t = allreduce_sum_(t).cpu()
        cross = float(t[0] / t[1]) if t[1] > 0 else None
        wait = float(t[2] / t[3]) if t[3] > 0 else None
        choice = float(t[4] / t[5]) if t[5] > 0 else float("nan")
        return cross, wait, choice, (int(t[1]), int(t[3]), int(t[5]))

    # -- checkpoints: same file names and state_dict layout as the reference (PY:935-1001) ------------------------
    _PATH = "load_model/weights/{stem}-{name}-{num_algo:02d}-{kind}-step-{epoch:03d}0.pth"

    def evaluate(self, nbr_episodes, choix=False, **kw):
        """Testing (PY:738-747): the deterministic rollout of every env for `nbr_episodes` episodes.  Returns the dense
        per-step records of Env_rollout.iterations; `self.rollout.reference_batches(out, n)` gives env n's
        (state_batch, action_batch, rew_c_batch, rew_d_batch, time_stop_batch) in the reference's shapes."""
        self.rollout.reset()
        return self.rollout.iterations(self.actor_net_cross, self.actor_net_wait, self.actor_net_choice, nbr_episodes, choix=choix, **kw)

    def evaluate_dataset(self, snapshot, **kw):
        """Testing on a stored scenario dataset (PY:749-758): one deterministic episode from every scenario of the snapshot file
        (the reference unpickles `test_data_23.pickle`, a list of deep-copied envs; here a VecCrosswalkEnv.save_state file)."""
        return self.rollout.iterations_dataset(self.actor_net_cross, self.actor_net_wait, self.actor_net_choice, snapshot, **kw)

    def _nets(self):
        return [("cross", "actor", self.actor_net_cross), ("wait", "actor", self.actor_net_wait), ("choice", "actor", self.actor_net_choice),
                ("cross", "critic", self.critic_net_cross), ("wait", "critic", self.critic_net_wait), ("choice", "critic", self.critic_net_choice)]

    def saving(self, root="."):
        for name, kind, net in self._nets():
            path = os.path.join(root, self._PATH.format(stem=self._STEM[self.env.variant], name=name, kind=kind, num_algo=self.num_algo, epoch=int(self.total_loop / 10)))
            os.makedirs(os.path.dirname(path), exist_ok=True)
            torch.save(net.state_dict(), path)

    def loading_curriculum(self, num_actor, num_algo, total_loop, root="."):
        """Load ONE (actor, critic) pair from another configuration's checkpoint (PY:957-984): num_actor 0 cross, 1 wait,
        2 choice; `num_algo` names the configuration the files were trained on (curriculum over nb_ped / nb_car / nb_lines)."""
        self.total_loop = total_loop
        name = {0: "cross", 1: "wait", 2: "choice"}[int(num_actor)]
        for n, kind, net in self._nets():
            if n == name:
                path = os.path.join(root, self._PATH.format(stem=self._STEM[self.env.variant], name=n, kind=kind, num_algo=num_algo,
                                                            epoch=int(total_loop / 10)))
                net.load_state_dict(torch.load(path, map_location="cpu"))
        self.sync_parameters()

    def loading(self, num_algo, total_loop, root="."):
        self.num_algo, self.total_loop = num_algo, total_loop
        for name, kind, net in self._nets():
            path = os.path.join(root, self._PATH.format(stem=self._STEM[self.env.variant], name=name, kind=kind, num_algo=num_algo, epoch=int(total_loop / 10)))
            net.load_state_dict(torch.load(path, map_location="cpu"))
        self.sync_parameters()
