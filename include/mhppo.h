/* mhppo.h -- C ABI of libmhppo_b200.so: the B200 (sm_100a) drop-in for MH-PPO's hot path.
 *
 * The reference (BrunoudA/MH-PPO) has no FFI: its seam is the gym-0.26 `Env` Python API of the six
 * `Environments/Env_hybrid_multi_*.py` classes plus the torch calls of `Env_rollout` / `Algo_PPO`
 * in `Coop-MH-PPO-scalable.py`.  Each entry point below names the reference interface it replaces
 * (file:line, abbreviations: SC = Environments/Env_hybrid_multi_coop_scalable.py, CO = .._coop.py,
 * ST = .._stop.py, NA = .._naif.py, C4 = .._coop_4cars.py, C42 = .._coop_4cars2.py,
 * PY = Coop-MH-PPO-scalable.py).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *  - plain C types only; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - every pointer named *_dev is device memory owned by the caller (e.g. torch tensor.data_ptr());
 *    the library never frees or retains it past the call; *_host pointers are host memory;
 *  - every call returns 0 on success or a negative MHPPO_E* code; mhppo_last_error() gives the text
 *    for the calling thread; nothing throws, nothing allocates after *_create;
 *  - all work is enqueued on `stream`, no hidden synchronisation (except the *_host entry points,
 *    which synchronise `stream` before returning because they fill host buffers);
 *  - one handle = one GPU = one host thread at a time.
 *  - there is NO CPU fallback: without a CUDA device every call fails with MHPPO_ENODEV.
 */
#ifndef MHPPO_H
#define MHPPO_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MHPPO_ABI_VERSION 1

enum { MHPPO_OK = 0, MHPPO_EINVAL = -1, MHPPO_ENODEV = -2, MHPPO_ECUDA = -3, MHPPO_ENOMEM = -4,
       MHPPO_EUNSUPPORTED = -5 };

/* env classes of the reference, Environments/__init__.py:3-41 */
enum { MHPPO_ENV_STOP = 0, MHPPO_ENV_NAIF = 1, MHPPO_ENV_COOP = 2, MHPPO_ENV_COOP_4CARS = 3,
       MHPPO_ENV_COOP_4CARS2 = 4, MHPPO_ENV_COOP_SCALABLE = 5 };

/* Constructor arguments of the env classes (SC:680: car_b, ped_b, cross_b, nb_car, nb_ped, nb_lines,
 * dt, max_episode, simulation) plus what a vectorised env needs (n_envs, RNG stream, device). */
typedef struct mhppo_env_cfg {
    int32_t variant;      /* MHPPO_ENV_* */
    int32_t nb_car, nb_ped, nb_lines;
    int32_t max_episode;  /* 80 in the drivers (PY:1026) */
    int32_t sin_model;    /* simulation == "sin" */
    int32_t device;       /* CUDA device ordinal */
    int32_t reserved;
    double dt;            /* 0.3 */
    double car_b[4];      /* row-major 2x2 */
    double ped_b[8];      /* row-major 2x4 */
    double cross_b[2];
    uint64_t seed;        /* Philox key (RNG contract: DESIGN.md "RNG") */
    int64_t n_envs;       /* envs held by this handle */
    int64_t env_id0;      /* global id of env 0: rank r of R passes r*n_envs so shards are disjoint streams */
} mhppo_env_cfg;

typedef struct mhppo_env_dims {
    int32_t n_slots;      /* car slots in state: nb_car | 2*nb_car (4cars*) | 2*nb_lines (scalable) */
    int32_t n_lead;       /* cars with a reward / reward_light entry */
    int32_t n_action;     /* action vector length, [acc.., light..] as in SC:798-802 / C42:809-811 */
    int32_t n_obs;        /* flat observation: keys in gym-0.26 Dict order car,(car_follow),env,ped */
    int32_t n_ped;
    int32_t done_step;    /* step index whose step() returns done (79 for dt=.3, max_episode=80) */
    int32_t reserved[2];
} mhppo_env_dims;

/* A 2-D fp32 view [n_envs, width] with element strides, so callers may keep either the gym layout
 * (env_stride = width, comp_stride = 1) or the coalesced device layout (env_stride = 1,
 * comp_stride = n_envs).  ptr == NULL means "not wanted" for outputs.  The observation views of
 * mhppo_env_step need 0 <= comp_stride < 2^31 (MHPPO_EINVAL otherwise). */
typedef struct mhppo_view {
    float *ptr;
    int64_t env_stride;
    int64_t comp_stride;
} mhppo_view;

int mhppo_abi_version(void);
const char *mhppo_last_error(void);
int mhppo_device_count(void);

/* gym.make(id, **cfg) / Crosswalk_hybrid_multi_*.__init__  (SC:680-736, REG:3-41) */
int mhppo_env_create(const mhppo_env_cfg *cfg, void **handle);
int mhppo_env_destroy(void *handle);
int mhppo_env_get_dims(void *handle, mhppo_env_dims *dims);

/* Crosswalk_hybrid_multi_*.reset  (SC:884-946, CO:838-892, ST:847, NA:829, C4:850-911, C42:866-927).
 * mask_dev: uint8[n_envs] or NULL (= all). obs receives the first observation of reset envs only. */
int mhppo_env_reset(void *handle, const uint8_t *mask_dev, mhppo_view obs_dev, void *stream);

/* State injection of the reference (fixed scenarios: choix_test PY:629-633, reset_distrib NA:903-913), for the envs with
 * mask_dev[n] != 0 (NULL = all).  One parameter row per env, device memory:
 *   reset_pedestrian (SC:948-955; CO:895, ST:904, C4:913, C42:929): params [N][9] = speed_x, speed_y, pos_x, pos_y, dl, leave, CZ,
 *     exist, direction.  Like the reference it first rebuilds EVERY pedestrian as a placeholder (their constructor draws are
 *     consumed from the env's stream), then applies pedestrian.reset_ped (SC:106-137) to slot num_ped; `leave` / `CZ` are stored
 *     as truth values.  naif (NA:897-898, 100-135): params = speed_x, speed_y, pos_x, pos_y, dl, direction, cross, -, - ; no
 *     rebuild; `cross` becomes the env's crossing width.
 *   reset_cars (SC:957-958 -> car.reset_car SC:583-587): params [N][4] = speed_x, pos_x, light, line (0 <= line < nb_lines: the
 *     kernels evaluate the lane predicates once per lane of the crossing).
 * Call mhppo_env_observe afterwards for the observation (the reference calls get_state(), PY:172-173). */
int mhppo_env_reset_pedestrian(void *handle, int32_t num_ped, const float *params_dev, const uint8_t *mask_dev, void *stream);
int mhppo_env_reset_cars(void *handle, int32_t num_car, const float *params_dev, const uint8_t *mask_dev, void *stream);

/* Crosswalk_hybrid_multi_*.get_state (SC:960-969): observation of the current state without stepping (after an
 * import_state / state injection).  As in the reference, get_data folds the current gap into every pedestrian's
 * running-min `delta` (SC:457), i.e. the call is not idempotent on that one field. */
int mhppo_env_observe(void *handle, mhppo_view obs_dev, void *stream);

/* Crosswalk_hybrid_multi_*.step  (SC:789-878, CO:745-832, ST:754, NA:736, C4:783-844, C42:799-860).
 * actions [n_envs,n_action]; obs [n_envs,n_obs]; rewards, reward_light (= env.reward_light, SC:846)
 * [n_envs,n_lead]; done uint8[n_envs].  autoreset != 0: a done env is re-initialised inside the same
 * kernel (gym vector convention): obs = first observation of the new episode, term_obs (optional) =
 * terminal observation. */
int mhppo_env_step(void *handle, mhppo_view actions_dev, mhppo_view obs_dev, mhppo_view rewards_dev,
                   mhppo_view reward_light_dev, uint8_t *done_dev, int autoreset, mhppo_view term_obs_dev,
                   void *stream);

/* Same call for HOST buffers in the reference's own layout (row-major [n_envs, width], what
 * env.step(np.ndarray) takes and returns): copies actions host->device, steps, copies the results
 * back and synchronises `stream`.  The env range is processed in slices on streams owned by the handle so that the
 * device->host copy of one slice overlaps the host->device copy and the kernel of the next; the device staging
 * buffers live in the handle, the host buffers are the caller's (pin them for full PCIe rate). */
int mhppo_env_step_host(void *handle, const float *actions_host, float *obs_host, float *rewards_host,
                        float *reward_light_host, uint8_t *done_host, int autoreset, void *stream);
int mhppo_env_reset_host(void *handle, float *obs_host, void *stream);

/* get_state()/reset_pedestrian()/reset_cars() of the reference read/poke Python attributes
 * (SC:948-969).  The vectorised equivalent moves the whole state as the canonical dump
 *   car_f [N,C,7] Ac,Vc,Sc,light,possible_accident,error_scenario,Ts      car_i [N,C,2] line,exist
 *   ped_f [N,P,9] Vp_x,Vp_y,Sp_x,Sp_y,v0x,v0y,cross_stop,delta,worst_dl
 *   ped_i [N,P,9] t0/dt,waiting_time/dt,crossing_time/dt,time_stop,line_pos,direction,gender,age,flags
 *   env_f [N,1]   cross (fp64)                env_i [N,4] step_idx,ped_traffic,car_traffic,rng_ctr
 * flags bits: 0 exist,1 is_crossing,2 decision,3 at_crossing,4 ped_left,5 ped_in_cross,
 * 6 ped_not_waiting,7 accident,8 worst_scenario_accident,9 follow_rule,10 stop,11 need_to_stop,
 * 12 ratio_eps (set by reset_ped: x follows y with ratio v0x / (v0y + 1e-3), SC:111, instead of v0x / v0y, SC:73).
 * All pointers are device memory. */
int mhppo_env_export_state(void *handle, float *car_f_dev, int32_t *car_i_dev, float *ped_f_dev,
                           int32_t *ped_i_dev, double *env_f_dev, int64_t *env_i_dev, void *stream);
int mhppo_env_import_state(void *handle, const float *car_f_dev, const int32_t *car_i_dev,
                           const float *ped_f_dev, const int32_t *ped_i_dev, const double *env_f_dev,
                           const int64_t *env_i_dev, void *stream);

/* bytes of HBM the handle holds per env (state arena), for the roofline accounting */
int64_t mhppo_env_state_bytes_per_env(void *handle);
/* number of kernel launches this library has issued in this process (bench.py "gpu_launches") */
int64_t mhppo_launch_count(void);

/* =====================================================================================================
 * PPO side: Model_PPO / Env_rollout / Algo_PPO of Coop-MH-PPO-scalable.py (scalable env class).
 *
 * Networks (Model_PPO, PY:42-93): in -> 32 -> 64 -> 32 -> out, ReLU; heads: 0 linear (critics),
 * 1 3*tanh(z)-1 (cross / wait actors, PY:1044-1045), 2 softmax over two logits (choice actor).
 * Flat parameter layout shared by every kernel (host packs/unpacks state_dicts):
 *   W1t[KP][32] b1[32] W2t[32][64] b2[64] W3t[64][32] b3[32] W4t[32][4] b4[4]   (weights transposed, zero padded;
 *   KP = mhppo_net_padded_in(n_in)).
 *
 * Buffers (device, fp32, env index innermost): obs [n_obs][N] (the env's component-major observation);
 * action_d int8 [C*P][N]; light [C][N]; sample s = (t*C + car)*N + env, S = T*C*N: obs_c [13][S], act, logp,
 * rew, rl, rtg, V [S]; choice sample m = car*N + env, M = C*N: obs_d [D][M], act_d, logp_d, rew_d [M];
 * route int8 [C][N] (0 cross, 1 wait, -1 car absent; PY:489-502).  C = 2*nb_lines, D = 2+6*(C-1)+10. */
typedef struct mhppo_rollout_cfg {
    int32_t nb_ped, nb_lines;
    int32_t T;            /* steps per episode (80) */
    int32_t legacy_nb_car; /* 0: Coop-MH-PPO-scalable.py layout (C = 2*nb_lines slots of 7 floats, env row of 4).  > 0: the older
                            * notebooks' layout on the coop / naif / stop env classes (Coop-MH-PPO.ipynb, MH-PPO.ipynb): C = this many
                            * cars of 6 floats, env row of 3, D = 2+5*(C-1)+10, every pedestrian slot visited, closest pedestrian
                            * seeded with slot 0 and not filtered on `exist` */
    int64_t n_envs;
    uint64_t seed;        /* same Philox key as the env */
    int64_t env_id0;
} mhppo_rollout_cfg;

/* Gaussian head of the cross / wait actors and its exploration noise, for the calling thread's later rollout / update calls:
 * mu = tanh(z) * std + mean (Model_PPO head type 1, PY:88-90; the driver derives mean = (car_b[1,0] + car_b[0,0]) / 2 and
 * std = (car_b[1,0] - car_b[0,0]) / 2, PY:1044-1045), a ~ N(mu, variance) (Algo_PPO.value_std, PY:726-729), acc_hi = car_b[1,0]
 * is the start value of the min over pedestrians (PY:436).  Defaults: -1, 3, 0.5, 2. */
int mhppo_set_gaussian_head(float mean, float std, float variance, float acc_hi);
int mhppo_net_padded_in(int32_t n_in);
int mhppo_net_param_count(int32_t n_in);

/* episode-start discrete decision of Env_rollout.iterations_rand (PY:400-428): obs_car_ped_d (PY:574-611) ->
 * choice net -> Categorical sample per (car, ped); closest_ped_d (PY:614-627) picks the car's light */
int mhppo_choice_act(const mhppo_rollout_cfg *cfg, const float *obs_dev, const float *net_choice_dev, uint32_t iteration,
                     int8_t *action_d_dev, float *light_dev, float *obs_d_dev, float *act_d_dev, float *logp_d_dev,
                     void *stream);
/* per-step continuous action (PY:434-453): obs_car_ped (PY:541-572) -> cross|wait net per pair -> min over existing
 * pedestrians -> N(mean, 0.5) sample + log-prob; writes the env's action buffer [2C][N] and the rollout buffers */
int mhppo_policy_act(const mhppo_rollout_cfg *cfg, const float *obs_dev, const float *net_cross_dev, const float *net_wait_dev,
                     const int8_t *action_d_dev, const float *light_dev, int32_t t, uint32_t iteration, float *actions_dev,
                     float *obs_c_dev, float *act_dev, float *logp_dev, void *stream);
/* The whole T-step inner loop of Env_rollout.iterations_rand (PY:386-476) in one call: per step policy_act, then env.step
 * with rewards / reward_light written into rew_dev / rl_dev [T][C][N] (no auto-reset: the episode ends at step T-1).
 * use_graph != 0: from the second call with the same arguments on, the 2T launches are replayed as one CUDA graph on a
 * stream owned by the library (launch-bound at small env counts); the caller's stream is ordered around it by events. */
int mhppo_rollout_steps(void *env_handle, const mhppo_rollout_cfg *cfg, float *obs_dev, const float *net_cross_dev,
                        const float *net_wait_dev, const int8_t *action_d_dev, const float *light_dev, uint32_t iteration,
                        float *actions_dev, float *obs_c_dev, float *act_dev, float *logp_dev, float *rew_dev, float *rl_dev,
                        uint8_t *done_dev, int32_t use_graph, void *stream);
/* deterministic evaluation rollout, Env_rollout.iterations (PY:152-252).
 * choice_eval: argmax of the choice net per (car, ped) (PY:177-192) for the envs that re-decide: all when force != 0 (first
 *   step of an episode), else those whose state has ped_traffic != nb_ped (PY:222-224); other envs keep action_d.
 * policy_eval: per car, min over ALL pedestrian slots of {net output | speed-recovery clip((speed_limit - v)/dt, acc_lo,
 *   acc_hi) when the pedestrian has left the lane}, capped by (10 - v)/dt (PY:195-214); writes the env's action buffer
 *   [2C][N] (lights = the first C entries of action_d, PY:192/216) and optionally the accelerations act_dev [C][N]. */
int mhppo_choice_eval(const mhppo_rollout_cfg *cfg, const float *obs_dev, const float *net_choice_dev, int32_t force,
                      int8_t *action_d_dev, void *stream);
int mhppo_policy_eval(const mhppo_rollout_cfg *cfg, const float *obs_dev, const float *net_cross_dev, const float *net_wait_dev,
                      const int8_t *action_d_dev, float dt, float speed_limit, float acc_lo, float acc_hi, float *actions_dev,
                      float *act_dev, void *stream);
/* Episode statistics of the evaluation records (the analysis cell get_average, PY:1550-1675, and the waiting-time histogram input
 * PY:1390-1403) on the device.  obs_rec: the dense record of Env_rollout.iterations, [E][T][n_obs][N] (state before each step).
 * ped_out [2][E][P][N]: waiting time on the kerb, crossing time, seconds (PY:1591-1601).  car_out [8][E][C][N]: time to 25 m past the
 * pedestrians (PY:1622-1631), free-flow time (25 - x0)/v0 (PY:1612), light at the last row (PY:1620), light after the first step
 * (PY:1613), could-stop flag (-1 if light1 >= 0, else 0 / 1, PY:1613-1617), number / sum / sum of squares of the 25 m passage times
 * (PY:1624-1625).  sums [E][N][8] = rows, sum v0, sum v0^2, sum |a0|, sum a0, sum a0^2, sum |vp0|, sum vp0^2 (PY:1552-1562);
 * yield_speed [E][N][3] = n, sum v, sum v^2 over the rows of cars with light1 == 1 (PY:1621).  The printed means / standard
 * deviations / scenario frequencies are reductions of these arrays (host mirror: Env_rollout.get_average). */
int mhppo_episode_stats(const float *obs_rec_dev, int32_t E, int32_t T, int32_t n_cars, int32_t n_ped, int32_t car_w, int32_t env_w,
                        int64_t N, float dt, float *ped_out_dev, float *car_out_dev, double *sums_dev, double *yield_speed_dev,
                        void *stream);
/* Env_rollout.futur_rewards (PY:658-684): reverse scan rtg_t = r_t + gamma*rtg_{t+1}, zero bootstrap; and the
 * episodic choice reward min(0, min_t reward_light) (PY:461).  CN = C*N */
int mhppo_returns(const float *rew_dev, const float *rl_dev, int32_t T, int64_t CN, double gamma, float *rtg_dev,
                  float *rew_d_dev, void *stream);

/* Algo_PPO.train_model_c / train_model_d (PY:778-851), one epoch = value_stats -> [all-reduce] -> ppo_grad (actor),
 * ppo_grad (critic) -> [all-reduce] -> adam.  x: features [D][S], sample slot s = t*CN + m.  idx: int32[K], the
 * compacted list of the (car, env) columns m routed to the net being trained (PY:489-502), NULL = all CN columns. */
int64_t mhppo_update_workspace_bytes(int32_t n_in);
int mhppo_value_stats(int32_t n_in, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K, int64_t CN,
                      const float *critic_dev, const float *rtg_dev, float *V_dev, double *stats3_dev, void *workspace_dev,
                      void *stream);
/* head: 0 critic MSE, 1 Gaussian actor clipped surrogate, 2 categorical actor (with the (M,M) broadcast of PY:834-842,
 * f0/f1 = fraction of selected samples whose action is 0/1).  grad_dev: flat gradient, loss_dev: fp64 scalar. */
int mhppo_ppo_grad(int32_t n_in, int32_t head, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K,
                   int64_t CN, const float *net_dev, const float *act_dev, const float *logp_old_dev, const float *rtg_dev,
                   const float *V_dev, float adv_mean, float adv_inv_std, float inv_n, float f0, float f1, float *grad_dev,
                   double *loss_dev, void *workspace_dev, void *stream);
/* mhppo_ppo_grad with the advantage statistics taken from DEVICE memory: adv_stats_dev = (sum A, sum A^2, n) over the whole batch
 * (the output of mhppo_critic_grad_stats, all-reduced over the ranks); mean and 1 / (unbiased std + 1e-10) (PY:787) are derived
 * inside the kernel, so an epoch needs no host round trip. */
int mhppo_ppo_grad_dev(int32_t n_in, int32_t head, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K,
                       int64_t CN, const float *net_dev, const float *act_dev, const float *logp_old_dev, const float *rtg_dev,
                       const float *V_dev, const double *adv_stats_dev, float inv_n, float f0, float f1, float *grad_dev,
                       double *loss_dev, void *workspace_dev, void *stream);
/* mhppo_ppo_grad_dev plus an entropy bonus for the categorical choice actor (an option; the reference's loss has none):
 * loss -= ent_coef * inv_n * sum_s H(pi(.|s)), H = -sum_k p_k log p_k over the two-way softmax, log p_k formed as log-softmax
 * (finite for saturated logits).  ent_coef == 0 runs exactly the kernel of mhppo_ppo_grad_dev (bit-identical results).
 * MHPPO_EINVAL for a non-finite ent_coef or a non-zero one with head != 2 (the Gaussian heads have a fixed variance: their
 * entropy is a constant without gradient). */
int mhppo_ppo_grad_ent(int32_t n_in, int32_t head, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K,
                       int64_t CN, const float *net_dev, const float *act_dev, const float *logp_old_dev, const float *rtg_dev,
                       const float *V_dev, const double *adv_stats_dev, float inv_n, float f0, float f1, float ent_coef,
                       float *grad_dev, double *loss_dev, void *workspace_dev, void *stream);
/* GAE(gamma, lambda) returns of the cross / wait buffers (an option; the reference's estimator is mhppo_returns, i.e. lambda = 1
 * with the critic recomputed every epoch).  Per column m of route_dev int8 [CN] (0 cross, 1 wait, -1 absent) over
 * t = T-1 .. 0 with V(s_T) = 0, R_T = 0, in fp64:  R_t = r_t + gamma ((1 - lambda) V(s_{t+1}) + lambda R_{t+1}),
 * ret_t = (float)R_t, A_t = ret_t - V(s_t) (fp32, as the actor forms it).  V_dev: V_old of the update (mhppo_value_stats of
 * each buffer's critic on its selection).  Absent columns get ret = 0 and are not read.  stats6_dev: (sum A, sum A^2, n) of
 * route 0, then of route 1, in a fixed summation order (bitwise repeatable); +0 / +3 are adv_stats_dev of the cross / wait
 * actor.  At lambda = 1 ret equals mhppo_returns' rtg bit for bit.  workspace_dev: 196 608 bytes (any update workspace of
 * mhppo_update_workspace_bytes is larger).  MHPPO_EINVAL for null pointers, T < 1, CN < 1, gamma or lambda outside [0, 1]. */
int mhppo_gae(const float *rew_dev, const float *V_dev, const int8_t *route_dev, int32_t T, int64_t CN, double gamma, double lambda,
              float *ret_dev, double *stats6_dev, void *workspace_dev, void *stream);
/* Minibatch plan of an update (an option, Algo_PPO(n_minibatches=B); the reference's update is full-batch, PY:866-882).
 * In epoch e (0 .. epochs-1) the (car, env) column m = car*N + n, global env id g = cfg->env_id0 + n, goes to bucket
 *   b = (x0 * B) >> 32,  x0 = word 0 of Philox4x32-10(counter = (e*C + car, 3 | iteration << 8, g_lo, g_hi), key = cfg->seed)
 * (stream 3 of the policy-noise contract; iteration = the rollout that filled the buffers), so a sharded run forms the same global
 * minibatches as one rank holding every env.  route_dev / exist_dev int8 [C][N], act_d_dev float [C*N] (choice actions 0 / 1).
 * Outputs, per epoch, for the selections s = 0 cross (route 0), 1 wait (route 1), 2 existing cars (exist != 0):
 *   lists_dev   int32 [epochs][3][C*N]: bucket-major column lists, ascending m within a bucket (at B = 1 the compacted lists of
 *               torch.nonzero); bucket b of selection s is lists[e][s][offsets[e][s][b] .. offsets[e][s][b+1])
 *   offsets_dev int64 [epochs][3][B+1]
 *   counts_dev  int64 [epochs][5][B]: bucket sizes of the three selections, then the existing columns whose choice action is 0 / 1
 * Integer counting sort in a fixed order (no order from atomics): repeated calls give identical outputs.  Three launches.
 * workspace_dev: 1280 * epochs * B bytes.  MHPPO_EINVAL for null pointers, epochs < 1, B outside [1, 1024] (the per-tile
 * histograms of five rows x B buckets live in 20 KB of shared memory), N < 1 or C*N >= 2^31. */
int mhppo_minibatch_plan(const mhppo_rollout_cfg *cfg, const int8_t *route_dev, const int8_t *exist_dev, const float *act_d_dev,
                         uint32_t iteration, int32_t epochs, int32_t n_minibatches, int32_t *lists_dev, int64_t *offsets_dev,
                         int64_t *counts_dev, void *workspace_dev, void *stream);
/* critic pass of one epoch in a single kernel: ppo_grad with head 0 that also returns V = critic(s) (PY:785) and the
 * advantage statistics (sum A, sum A^2, n) of A = rtg - V, so an epoch is critic_grad_stats -> [all-reduce stats] ->
 * ppo_grad (actor) -> [all-reduce grads] -> adam, adam; V and the statistics are those of the critic before its step,
 * as in the reference (the actor and critic steps of PY:810-815 act on different networks).  inv_n = 1 / global count */
int mhppo_critic_grad_stats(int32_t n_in, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K, int64_t CN,
                            const float *critic_dev, const float *rtg_dev, float inv_n, float *grad_dev, double *loss_dev,
                            float *V_dev, double *stats3_dev, void *workspace_dev, void *stream);
/* torch.optim.Adam defaults (PY:719-724); step counts from 1; grad_scale multiplies the gradient first */
int mhppo_adam(float *param_dev, const float *grad_dev, float *m_dev, float *v_dev, int32_t n, float lr, float beta1,
               float beta2, float eps, int32_t step, float grad_scale, void *stream);

/* the actor's and the critic's Adam step of one epoch in one launch (they act on different nets, PY:810-815) */
int mhppo_adam2(float *p0_dev, const float *g0_dev, float *m0_dev, float *v0_dev, int32_t n0, float lr0, int32_t step0, float *p1_dev,
                const float *g1_dev, float *m1_dev, float *v1_dev, int32_t n1, float lr1, int32_t step1, float beta1, float beta2,
                float eps, void *stream);

/* Update diagnostics (an option, Algo_PPO(diagnostics=True) / Algo_PPO(target_kl=delta); the reference logs nothing about its
 * update).  The two passes below are mhppo_critic_grad_stats / mhppo_ppo_grad (head 0, GAE mode) and mhppo_ppo_grad_ent with the
 * same gradient, loss and statistics outputs bit for bit; in the same kernel pass they also sum, per step (one Adam step of a pair),
 * over this rank's samples, at the parameters before the step, and write into the step's RECORD ROW (fp64 [10], caller-zeroed):
 *   [0] actor loss  [1] critic loss  (the values loss_dev receives)
 *   [2] sum k3 = r - 1 - log r, log r = log pi(a_s|s) - logp_old[s] (Gaussian heads: the loss's log-prob; choice head: the
 *       log-softmax of the TAKEN action act_dev[s]), fp32 log r, k3 in fp64 as expm1(log r) - log r
 *   [3] count of r < 0.8 or r > 1.2 on the fp32 ratio the loss's clamp sees (choice: p_a * exp(-logp_old))
 *   [4] sum H(pi(.|s)) (head 2 only, log-softmax form; 0 otherwise)
 *   [5] sum (R - V)  [6] sum (R - V)^2  [7] sum R  [8] sum R^2   (R = rtg_dev, the critic's target; V = this pass's forward)
 *   [9] taken: 1.0 once mhppo_adam2_halt (or mhppo_adam2_clip with the halt) takes the step (written by nothing else)
 * Per-CTA fp64 partials, reduced in a fixed order by one more kernel per pass (no floating-point atomics): repeatable bit for
 * bit.  Ratios (approx_kl = [2] / n, clip fraction = [3] / n, entropy = [4] / n, explained variance = 1 - Var(R-V) / Var(R)) are
 * formed by the caller from the sums over all ranks.
 * critic_grad_diag: V_dev and stats3_dev both given = mhppo_critic_grad_stats; both NULL = the critic pass of GAE mode, which does
 * not write V. */
int mhppo_critic_grad_diag(int32_t n_in, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K, int64_t CN,
                           const float *critic_dev, const float *rtg_dev, float inv_n, float *grad_dev, double *loss_dev,
                           float *V_dev, double *stats3_dev, double *record_row_dev, void *workspace_dev, void *stream);
/* ppo_grad_diag: the actor pass (head 1 or 2) of mhppo_ppo_grad_ent with the diagnostics above; kl_slot_dev (may be NULL) receives
 * record[2] as fp32 -- place it behind the pair's packed gradients so that the gradient all-reduce also sums it over the ranks. */
int mhppo_ppo_grad_diag(int32_t n_in, int32_t head, const float *x_dev, int32_t D, int64_t S, const int32_t *idx_dev, int64_t K,
                        int64_t CN, const float *net_dev, const float *act_dev, const float *logp_old_dev, const float *rtg_dev,
                        const float *V_dev, const double *adv_stats_dev, float inv_n, float f0, float f1, float ent_coef,
                        float *grad_dev, double *loss_dev, float *kl_slot_dev, double *record_row_dev, void *workspace_dev,
                        void *stream);
/* mhppo_adam2 with the target-KL halt of SB3, checked before the step: if *halt_dev != 0 (int32, zeroed by the caller at the start of
 * an update) nothing happens; else if *kl_sum_dev (the all-reduced fp32 k3 sum of the step) > kl_limit (= 1.5 * target_kl * n) the
 * step is not taken and *halt_dev = 1, so every later launch with this flag does nothing; else both Adam steps are taken, with
 * mhppo_adam2's arithmetic, and record_row_dev[9] = 1.0.  No host round trip. */
int mhppo_adam2_halt(float *p0_dev, const float *g0_dev, float *m0_dev, float *v0_dev, int32_t n0, float lr0, int32_t step0, float *p1_dev,
                     const float *g1_dev, float *m1_dev, float *v1_dev, int32_t n1, float lr1, int32_t step1, float beta1, float beta2,
                     float eps, const float *kl_sum_dev, double kl_limit, int32_t *halt_dev, double *record_row_dev, void *stream);

/* mhppo_adam2 with per-network gradient-norm clipping (an option, Algo_PPO(max_grad_norm=g); the reference does not clip), torch's
 * clip_grad_norm_(net.parameters(), max_norm) before each net's step: norm = the fp64 L2 norm of the net's whole flat gradient
 * (n0 / n1 floats; the padded slots of the flat layout are exactly 0 after every gradient pass, so it is the norm over the
 * reference-layout tensors), coef = max_norm / (norm + 1e-6), and the Adam step uses coef * grad when coef < 1, else the gradient
 * unchanged.  A non-finite norm gives coef = 1.  An unclipped step is mhppo_adam2's (mhppo_adam2_halt's) bit for bit; g0_dev and
 * g1_dev are not written.  norms_out_dev (may be NULL): fp64 [2], actor (net 0) then critic (net 1).  kl_sum_dev, kl_limit, halt_dev,
 * record_row_dev: mhppo_adam2_halt's halt, tested after the norms are written (a halted step still reports its norms); all three
 * pointers NULL = no halt, kl_limit unused.  Sum of squares in a fixed order (no atomics): repeatable bit for bit.  One launch.
 * MHPPO_EINVAL: mhppo_adam2's checks, max_norm NaN or <= 0 (+inf records the norms and never clips), some but not all halt
 * pointers, kl_limit NaN with the halt. */
int mhppo_adam2_clip(float *p0_dev, const float *g0_dev, float *m0_dev, float *v0_dev, int32_t n0, float lr0, int32_t step0, float *p1_dev,
                     const float *g1_dev, float *m1_dev, float *v1_dev, int32_t n1, float lr1, int32_t step1, float beta1, float beta2,
                     float eps, double max_norm, double *norms_out_dev, const float *kl_sum_dev, double kl_limit, int32_t *halt_dev,
                     double *record_row_dev, void *stream);

/* mhppo_adam2_clip with the KL-adaptive learning rate (an option, Algo_PPO(lr_schedule="adaptive", desired_kl=delta); rsl_rl's
 * schedule="adaptive" rule, decided on the device before the step): kl = *kl_sum_dev / n, the pair's all-reduced actor k3 sum (the
 * fp32 slot mhppo_ppo_grad_diag writes behind the pair's packed gradients) over the step's sample count n; then on each net's fp32 lr
 * state lr_dev[0] (actor, net 0) and lr_dev[1] (critic, net 1) separately:
 *   kl > 2 delta            lr = max(1e-5, lr / 1.5)
 *   0 < kl < delta / 2      lr = min(1e-2, lr * 1.5)
 *   otherwise (NaN, +-inf)  lr unchanged
 * each change computed in fp64 and rounded to fp32.  The step uses that lr: step size (float)((double)lr / (1 - beta1^step)), the
 * formula of mhppo_adam2, so a step whose lr did not change is mhppo_adam2_clip's (mhppo_adam2's when nothing is clipped) bit for bit.
 * lr0 and lr1 are unused.  lrs_out_dev (may be NULL): fp64 [2], the lrs the step used.  With the halt (kl_sum, halt_dev, record_row_dev)
 * its test comes first: a halted step changes neither the weights nor lr_dev nor lrs_out_dev.  max_norm = +inf: no clipping.  One launch.
 * MHPPO_EINVAL: mhppo_adam2_clip's checks, lr_dev or kl_sum_dev NULL, desired_kl NaN or <= 0, n NaN or <= 0. */
int mhppo_adam2_sched(float *p0_dev, const float *g0_dev, float *m0_dev, float *v0_dev, int32_t n0, float lr0, int32_t step0, float *p1_dev,
                      const float *g1_dev, float *m1_dev, float *v1_dev, int32_t n1, float lr1, int32_t step1, float beta1, float beta2,
                      float eps, double max_norm, double *norms_out_dev, const float *halt_kl_sum_dev, double kl_limit, int32_t *halt_dev,
                      double *record_row_dev, float *lr_dev, const float *kl_sum_dev, double n, double desired_kl, double *lrs_out_dev,
                      void *stream);

/* Self-test of the tcgen05 / TMEM building blocks behind the policy GEMMs: D[128,N] = A[128,K] * B[N,K]^T on one CTA,
 * mode 0 = one tf32 pass, mode 1 = 3xTF32 split accumulation.  (N,K) in {(64,32),(32,64),(64,16),(16,32)}. */
/* implementation of the 13-input nets' kernels: 0 auto (tcgen05 for the update: forward + backward-data of ppo_grad /
 * critic_grad_stats and the critic forward of value_stats; exact-fp32 FFMA for the rollout inference), 1 FFMA everywhere
 * (exact fp32 cross-check), 2 tcgen05 wherever a tensor-core kernel exists (also the rollout inference) */
int mhppo_set_mlp_mode(int32_t mode);
/* 1 if a tensor-core kernel ever timed out waiting for its MMAs (diagnostic; synchronises the device) */
int mhppo_tc_failures(void);
/* Self-test of the step kernel's gap-acceptance predicate (`car_time + light < CG`, SC:167-170, 419-428): for n samples
 * (device arrays) returns the filtered decision the kernel takes (fast), the level that took it (0 = no draw needed,
 * 1 = fp32 draw, 2 = exact fallback), the exact fp64 decision and the exact critical gap (cg_dev may be NULL).  The normal
 * draw of sample i is Philox block ctr[i] of stream (env_id, key0, key1).  fast must equal exact for every input. */
int mhppo_gap_selftest(int64_t n, const double *dx_dev, const double *vden_dev, const double *light_dev, const double *size_dev,
                       const double *v0y_dev, const int32_t *gender_dev, const int32_t *age_dev, const uint32_t *ctr_dev,
                       uint64_t env_id, uint32_t key0, uint32_t key1, uint8_t *fast_dev, uint8_t *level_dev, uint8_t *exact_dev,
                       double *cg_dev, void *stream);
int mhppo_tc_selftest(const float *A_dev, const float *B_dev, float *D_dev, int32_t N, int32_t K, int32_t mode, void *stream);

#ifdef __cplusplus
}
#endif
#endif
