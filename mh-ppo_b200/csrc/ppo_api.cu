// ppo_api.cu -- host side of the PPO part of the C ABI (include/mhppo.h).
#include <cmath>
#include <cstdio>
#include <string>

#include "../../include/mhppo.h"
#include "ppo_rollout.cuh"
#include "ppo_update.cuh"
#include "tc_kernels.cuh"
#include "tc_grad.cuh"
#include "stats.cuh"
#include <cstdlib>
#include <cstring>

namespace mhppo {
int api_fail(int code, const std::string &msg);      // mhppo_api.cu
void api_count_launch();
static int ck(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return 0;
    return api_fail(MHPPO_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
static int padded_in(int n_in) { return n_in <= 16 ? 16 : (n_in <= 32 ? 32 : (n_in <= 56 ? 56 : -1)); }
// Which implementation serves the 13-input nets' forward-only kernels (mhppo_set_mlp_mode):
//   0 auto : tcgen05 for the critic forward of the update (faster), FFMA for the rollout's per-step inference (the
//            tensor-core version of that kernel is latency-bound with one tile in flight per CTA, DESIGN.md "Kernels")
//   1 ffma : exact-fp32 CUDA-core kernels everywhere (cross-check)      2 tc : tcgen05 wherever a kernel exists
static int g_mlp_mode = []() { const char *e = std::getenv("MHPPO_MLP"); return (e && std::string(e) == "ffma") ? 1 : ((e && std::string(e) == "tc") ? 2 : 0); }();
static bool use_tc(bool rollout) { return g_mlp_mode == 2 || (g_mlp_mode == 0 && !rollout); }
static HeadCfg make_head(double mean, double std, double variance, double acc_hi) {
    HeadCfg h;
    h.mean = (float)mean; h.std = (float)std; h.sigma = (float)std::sqrt(variance); h.inv_2var = (float)(1.0 / (2.0 * variance));
    h.logp_c = (float)(0.5 * std::log(2.0 * 3.141592653589793 * variance)); h.acc_hi = (float)acc_hi;
    return h;
}
static thread_local HeadCfg g_head = make_head(-1.0, 3.0, 0.5, 2.0);      // PY:1044-1045, 726
// sticky per-device flag the tensor-core kernels raise when an mbarrier wait times out (their results are then
// unusable); Algo_PPO.update reads it through mhppo_tc_failures after every update and raises.  The PPO entry
// points have no handle, so the 4 bytes are allocated on the first tensor-core launch on each device.
static int *fail_flag() {
    static int *p[64] = {nullptr};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (!p[dev]) { cudaMalloc(&p[dev], sizeof(int)); cudaMemset(p[dev], 0, sizeof(int)); }
    return p[dev];
}
static size_t smem_tc(int nets) {
    return sizeof(float) * ((size_t)nets * ((tcm::NetTiles<16>::FLOATS + 255) & ~255) + 2 * 128 * H2) + 1024;
}
constexpr int kGradGridMax = 148;    // k_ppo_grad: one persistent CTA per SM (its tile fills shared memory); B200 has 148 SMs
constexpr int kUpdateGridMax = 296;  // rows of the partial buffers in the workspace: 2 per SM (CTAs of k_value_stats)
// grids follow the SM count of the current device (a smaller part runs fewer persistent CTAs, never more than the workspace holds)
static int sm_count() {
    static int n[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (!n[dev]) { int v = 0; cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); n[dev] = v > 0 ? v : kGradGridMax; }
    return n[dev];
}
static int grad_grid() { const int n = sm_count(); return n < kGradGridMax ? n : kGradGridMax; }
static int update_grid() { const int n = 2 * sm_count(); return n < kUpdateGridMax ? n : kUpdateGridMax; }
#define kGradGrid grad_grid()
#define kUpdateGrid update_grid()

template <int KP> static size_t smem_fwd(int nets) {
    return sizeof(float) * ((size_t)nets * ((net_params(KP) + 3) & ~3) + (size_t)kFwdBlock * kRowFwd);
}
template <int KP> static size_t smem_grad() {
    return sizeof(float) * GradCfg<KP>::smem_floats;
}
static RolloutDims dims_of(const mhppo_rollout_cfg *c) {
    RolloutDims d;
    d.P = c->nb_ped; d.L = c->nb_lines;
    d.legacy = c->legacy_nb_car > 0 ? 1 : 0;
    d.C = d.legacy ? c->legacy_nb_car : 2 * c->nb_lines;
    d.car_w = d.legacy ? 6 : 7; d.env_w = d.legacy ? 3 : 4;
    d.n_obs = d.car_w * d.C + d.env_w + 9 * d.P; d.D = 2 + (d.legacy ? 5 : 6) * (d.C - 1) + 10;
    d.N = c->n_envs; d.k0 = (uint32_t)c->seed; d.k1 = (uint32_t)(c->seed >> 32); d.env_id0 = c->env_id0;
    d.head = g_head;
    return d;
}
struct Workspace { float *gpartial; double *lpartial; double *spartial; double *dpartial; };
static Workspace carve(void *ws, int KP) {
    Workspace w;
    w.gpartial = (float *)ws;
    size_t off = sizeof(float) * (size_t)kUpdateGridMax * net_params(KP);
    off = (off + 15) & ~(size_t)15;
    w.lpartial = (double *)((char *)ws + off);
    w.spartial = w.lpartial + kUpdateGridMax;
    w.dpartial = w.spartial + (size_t)kUpdateGridMax * 3;      // [grid][kDiagW], the DIAG instances only
    return w;
}
}  // namespace mhppo

using namespace mhppo;

#define SET_SMEM(kernel, bytes)                                                                                      \
    do {                                                                                                             \
        int rc_ = ck(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)), #kernel); \
        if (rc_) return rc_;                                                                                         \
    } while (0)

// 13-input nets, heads 0 / 1: forward and backward-data on the tensor cores (tc_grad.cuh) unless MHPPO_MLP=ffma
template <bool DIAG>
static int launch_grad_tc(int head, const SampleSet &ss, const float *net, const LossArgs &la, const Workspace &w, cudaStream_t s) {
    const size_t sm = sizeof(float) * kTcGradSmemFloats;
    if (head == 0) { SET_SMEM((k_ppo_grad_tc<0, DIAG>), sm); k_ppo_grad_tc<0, DIAG><<<kGradGrid, kTcGradBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial, fail_flag()); }
    else { SET_SMEM((k_ppo_grad_tc<1, DIAG>), sm); k_ppo_grad_tc<1, DIAG><<<kGradGrid, kTcGradBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial, fail_flag()); }
    api_count_launch();
    return ck(cudaGetLastError(), "k_ppo_grad_tc");
}

template <int KP, bool DIAG>
static int launch_grad(int head, const SampleSet &ss, const float *net, const LossArgs &la, const Workspace &w, cudaStream_t s) {
    // (the tensor-core kernel stages exactly the 13 features of the cross / wait nets; a wider 16-padded input takes the FFMA kernel)
    if (KP == 16 && ss.D <= 13 && head != 2 && use_tc(false)) return launch_grad_tc<DIAG>(head, ss, net, la, w, s);
    const size_t sm = smem_grad<KP>();
    if (head == 2 && la.ent_coef != 0.f) { SET_SMEM((k_ppo_grad<KP, 2, true, DIAG>), sm); k_ppo_grad<KP, 2, true, DIAG><<<kGradGrid, kMlpBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial); }
    else if (head == 0) { SET_SMEM((k_ppo_grad<KP, 0, false, DIAG>), sm); k_ppo_grad<KP, 0, false, DIAG><<<kGradGrid, kMlpBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial); }
    else if (head == 1) { SET_SMEM((k_ppo_grad<KP, 1, false, DIAG>), sm); k_ppo_grad<KP, 1, false, DIAG><<<kGradGrid, kMlpBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial); }
    else { SET_SMEM((k_ppo_grad<KP, 2, false, DIAG>), sm); k_ppo_grad<KP, 2, false, DIAG><<<kGradGrid, kMlpBlock, sm, s>>>(ss, net, la, w.gpartial, w.lpartial); }
    api_count_launch();
    return ck(cudaGetLastError(), "k_ppo_grad");
}

extern "C" {

int mhppo_net_padded_in(int32_t n_in) { return padded_in(n_in); }
int mhppo_net_param_count(int32_t n_in) { const int kp = padded_in(n_in); return kp < 0 ? -1 : net_params(kp); }

int mhppo_choice_act(const mhppo_rollout_cfg *cfg, const float *obs, const float *net, uint32_t iteration, int8_t *action_d,
                     float *light, float *obs_d, float *act_d, float *logp_d, void *stream) {
    if (!cfg || !obs || !net || !action_d || !light || !obs_d || !act_d || !logp_d) return api_fail(MHPPO_EINVAL, "null argument");
    const RolloutDims d = dims_of(cfg);
    const int kp = padded_in(d.D);
    if (kp < 0) return api_fail(MHPPO_EUNSUPPORTED, "choice features wider than 56 (nb_lines > 4)");
    const dim3 grid((unsigned)((d.N + kFwdBlock - 1) / kFwdBlock), (unsigned)d.C);
    cudaStream_t s = (cudaStream_t)stream;
    if (kp == 16) { SET_SMEM(k_choice_act<16>, smem_fwd<16>(1)); k_choice_act<16><<<grid, kFwdBlock, smem_fwd<16>(1), s>>>(d, obs, net, iteration, action_d, light, obs_d, act_d, logp_d); }
    else if (kp == 32) { SET_SMEM(k_choice_act<32>, smem_fwd<32>(1)); k_choice_act<32><<<grid, kFwdBlock, smem_fwd<32>(1), s>>>(d, obs, net, iteration, action_d, light, obs_d, act_d, logp_d); }
    else { SET_SMEM(k_choice_act<56>, smem_fwd<56>(1)); k_choice_act<56><<<grid, kFwdBlock, smem_fwd<56>(1), s>>>(d, obs, net, iteration, action_d, light, obs_d, act_d, logp_d); }
    api_count_launch();
    return ck(cudaGetLastError(), "k_choice_act");
}

static int policy_act_impl(const mhppo_rollout_cfg *cfg, const float *obs, const float *net_cross, const float *net_wait,
                           const int8_t *action_d, const float *light, int32_t t, uint32_t iteration, const uint32_t *iter_dev,
                           float *actions, float *obs_c, float *act, float *logp, void *stream) {
    if (!cfg || !obs || !net_cross || !net_wait || !action_d || !light || !actions || !obs_c || !act || !logp)
        return api_fail(MHPPO_EINVAL, "null argument");
    const RolloutDims d = dims_of(cfg);
    ActIO io; io.obs = obs; io.action_d = action_d; io.light = light; io.actions = actions; io.obs_c = obs_c; io.act = act;
    io.logp = logp; io.t = t; io.T = cfg->T; io.iteration = iteration; io.iter_dev = iter_dev;
    if (use_tc(true)) {
        const int64_t items = ((d.N + 127) / 128) * d.C;
        const unsigned g2 = (unsigned)(items < sm_count() ? items : sm_count());       // persistent: one CTA per SM walks the (env block, car) items
        SET_SMEM(k_policy_act_tc, smem_tc(2));
        k_policy_act_tc<<<g2, 128, smem_tc(2), (cudaStream_t)stream>>>(d, net_cross, net_wait, io, fail_flag());
        api_count_launch();
        return ck(cudaGetLastError(), "k_policy_act_tc");
    }
    const dim3 grid((unsigned)((d.N + kFwdBlock - 1) / kFwdBlock), (unsigned)d.C);
    if (d.P > kActMaxP) return api_fail(MHPPO_EUNSUPPORTED, "more than 4 pedestrian slots");
    const size_t sm_act = smem_fwd<16>(2) + sizeof(float) * kFwdBlock * kActMaxP + sizeof(uint16_t) * kFwdBlock * kActMaxP;
    SET_SMEM(k_policy_act, sm_act);
    k_policy_act<<<grid, kFwdBlock, sm_act, (cudaStream_t)stream>>>(d, net_cross, net_wait, io);
    api_count_launch();
    return ck(cudaGetLastError(), "k_policy_act");
}

int mhppo_policy_act(const mhppo_rollout_cfg *cfg, const float *obs, const float *net_cross, const float *net_wait,
                     const int8_t *action_d, const float *light, int32_t t, uint32_t iteration, float *actions, float *obs_c,
                     float *act, float *logp, void *stream) {
    return policy_act_impl(cfg, obs, net_cross, net_wait, action_d, light, t, iteration, nullptr, actions, obs_c, act, logp, stream);
}

/* The T-step inner loop of Env_rollout.iterations_rand (PY:386-476) in one call: per step policy_act -> env.step, rewards and
 * reward_light written straight into the rollout buffers.  160 launches per episode are launch-bound for small env counts
 * (configs[1]: 4096 envs), so from the second call with the same arguments on the loop is replayed as ONE CUDA graph on a
 * stream owned by this library (the iteration number of the noise contract is read from device memory by the graph's
 * kernels); the caller's stream is ordered before and after it with events. */
namespace {
struct RolloutGraph {
    void *env; mhppo_rollout_cfg cfg; const void *p[12]; HeadCfg head; int mlp_mode;
    cudaGraphExec_t exec; cudaStream_t s; cudaEvent_t ev_in, ev_out; uint32_t *iter_dev; int calls;
};
static RolloutGraph g_rg = {};
}
// called by mhppo_env_destroy: a captured graph holds the env's arena pointers by value and must not outlive the handle
// (a later handle may be allocated at the same address)
}   // extern "C"
namespace mhppo { void rollout_forget_env(void *env) {
    if (g_rg.env == env) {
        if (g_rg.exec) { cudaGraphExecDestroy(g_rg.exec); g_rg.exec = nullptr; }
        g_rg.env = nullptr; g_rg.calls = 0;
    }
} }
extern "C" {

int mhppo_rollout_steps(void *env, const mhppo_rollout_cfg *cfg, float *obs, const float *net_cross, const float *net_wait,
                        const int8_t *action_d, const float *light, uint32_t iteration, float *actions, float *obs_c, float *act,
                        float *logp, float *rew, float *rl, uint8_t *done, int32_t use_graph, void *stream) {
    if (!env || !cfg || !obs || !rew || !rl || !done) return api_fail(MHPPO_EINVAL, "null argument");
    const RolloutDims d = dims_of(cfg);
    const int64_t N = d.N;
    const int T = cfg->T, Cn = d.C;
    cudaStream_t caller = (cudaStream_t)stream;
    auto run = [&](cudaStream_t q, const uint32_t *iter_dev) -> int {
        const mhppo_view none = { nullptr, 0, 0 };
        for (int t = 0; t < T; ++t) {
            int rc = policy_act_impl(cfg, obs, net_cross, net_wait, action_d, light, t, iteration, iter_dev, actions, obs_c, act, logp, q);
            if (rc) return rc;
            const int64_t off = (int64_t)t * Cn * N;
            rc = mhppo_env_step(env, mhppo_view{ actions, 1, N }, mhppo_view{ obs, 1, N }, mhppo_view{ rew + off, 1, N },
                                mhppo_view{ rl + off, 1, N }, done, 0, none, q);
            if (rc) return rc;
        }
        return 0;
    };
    if (!use_graph) return run(caller, nullptr);
    RolloutGraph &g = g_rg;
    const void *key[12] = { obs, net_cross, net_wait, action_d, light, actions, obs_c, act, logp, rew, rl, done };
    const bool same = g.exec && g.env == env && !memcmp(&g.cfg, cfg, sizeof(*cfg)) && !memcmp(g.p, key, sizeof(key)) &&
                      !memcmp(&g.head, &g_head, sizeof(HeadCfg)) && g.mlp_mode == g_mlp_mode;
    if (!g.s) {
        if (ck(cudaStreamCreateWithFlags(&g.s, cudaStreamNonBlocking), "cudaStreamCreate")) return MHPPO_ECUDA;
        cudaEventCreateWithFlags(&g.ev_in, cudaEventDisableTiming); cudaEventCreateWithFlags(&g.ev_out, cudaEventDisableTiming);
        if (ck(cudaMalloc(&g.iter_dev, sizeof(uint32_t)), "cudaMalloc")) return MHPPO_ECUDA;
    }
    if (!same) {
        // first call with these arguments: plain launches (they also set the kernels' shared-memory attributes), then capture
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
        g.env = env; g.cfg = *cfg; memcpy(g.p, key, sizeof(key)); g.head = g_head; g.mlp_mode = g_mlp_mode; g.calls = 0;
    }
    if (g.calls++ == 0) return run(caller, nullptr);
    if (ck(cudaEventRecord(g.ev_in, caller), "cudaEventRecord") || ck(cudaStreamWaitEvent(g.s, g.ev_in, 0), "cudaStreamWaitEvent")) return MHPPO_ECUDA;
    if (ck(cudaMemcpyAsync(g.iter_dev, &iteration, sizeof(uint32_t), cudaMemcpyHostToDevice, g.s), "cudaMemcpyAsync")) return MHPPO_ECUDA;
    if (!g.exec) {
        cudaGraph_t graph = nullptr;
        if (ck(cudaStreamBeginCapture(g.s, cudaStreamCaptureModeThreadLocal), "cudaStreamBeginCapture")) return MHPPO_ECUDA;
        const int rc = run(g.s, g.iter_dev);
        const cudaError_t e = cudaStreamEndCapture(g.s, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ck(e, "cudaStreamEndCapture")) return MHPPO_ECUDA;
        const cudaError_t e2 = cudaGraphInstantiate(&g.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ck(e2, "cudaGraphInstantiate")) { g.exec = nullptr; return MHPPO_ECUDA; }
    }
    if (ck(cudaGraphLaunch(g.exec, g.s), "cudaGraphLaunch")) return MHPPO_ECUDA;
    for (int k = 0; k < 2 * T; ++k) api_count_launch();           // the graph's kernel nodes
    if (ck(cudaEventRecord(g.ev_out, g.s), "cudaEventRecord") || ck(cudaStreamWaitEvent(caller, g.ev_out, 0), "cudaStreamWaitEvent")) return MHPPO_ECUDA;
    return 0;
}

int mhppo_choice_eval(const mhppo_rollout_cfg *cfg, const float *obs, const float *net, int32_t force, int8_t *action_d, void *stream) {
    if (!cfg || !obs || !net || !action_d) return api_fail(MHPPO_EINVAL, "null argument");
    const RolloutDims d = dims_of(cfg);
    const int kp = padded_in(d.D);
    if (kp < 0) return api_fail(MHPPO_EUNSUPPORTED, "choice features wider than 56 (nb_lines > 4)");
    const dim3 grid((unsigned)((d.N + kFwdBlock - 1) / kFwdBlock), (unsigned)d.C);
    cudaStream_t s = (cudaStream_t)stream;
    if (kp == 16) { SET_SMEM(k_choice_eval<16>, smem_fwd<16>(1)); k_choice_eval<16><<<grid, kFwdBlock, smem_fwd<16>(1), s>>>(d, obs, net, force, action_d); }
    else if (kp == 32) { SET_SMEM(k_choice_eval<32>, smem_fwd<32>(1)); k_choice_eval<32><<<grid, kFwdBlock, smem_fwd<32>(1), s>>>(d, obs, net, force, action_d); }
    else { SET_SMEM(k_choice_eval<56>, smem_fwd<56>(1)); k_choice_eval<56><<<grid, kFwdBlock, smem_fwd<56>(1), s>>>(d, obs, net, force, action_d); }
    api_count_launch();
    return ck(cudaGetLastError(), "k_choice_eval");
}

int mhppo_policy_eval(const mhppo_rollout_cfg *cfg, const float *obs, const float *net_cross, const float *net_wait,
                      const int8_t *action_d, float dt, float speed_limit, float acc_lo, float acc_hi, float *actions, float *act,
                      void *stream) {
    if (!cfg || !obs || !net_cross || !net_wait || !action_d || !actions) return api_fail(MHPPO_EINVAL, "null argument");
    if (!(dt > 0.f)) return api_fail(MHPPO_EINVAL, "dt must be > 0");
    const RolloutDims d = dims_of(cfg);
    if (d.P < 1 || (int64_t)d.C * d.P < d.C) return api_fail(MHPPO_EINVAL, "needs at least one pedestrian slot");
    EvalIO io; io.obs = obs; io.action_d = action_d; io.actions = actions; io.act = act;
    io.dt = dt; io.speed_limit = speed_limit; io.acc_lo = acc_lo; io.acc_hi = acc_hi;
    const dim3 grid((unsigned)((d.N + kFwdBlock - 1) / kFwdBlock), (unsigned)d.C);
    SET_SMEM(k_policy_eval, smem_fwd<16>(2));
    k_policy_eval<<<grid, kFwdBlock, smem_fwd<16>(2), (cudaStream_t)stream>>>(d, net_cross, net_wait, io);
    api_count_launch();
    return ck(cudaGetLastError(), "k_policy_eval");
}

int mhppo_returns(const float *rew, const float *rl, int32_t T, int64_t CN, double gamma, float *rtg, float *rew_d, void *stream) {
    if (!rew || !rl || !rtg || !rew_d) return api_fail(MHPPO_EINVAL, "null argument");
    k_returns<<<(unsigned)((CN + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rew, rl, T, CN, gamma, rtg, rew_d);
    api_count_launch();
    return ck(cudaGetLastError(), "k_returns");
}

int mhppo_episode_stats(const float *obs_rec, int32_t E, int32_t T, int32_t n_cars, int32_t n_ped, int32_t car_w, int32_t env_w, int64_t N,
                        float dt, float *ped_out, float *car_out, double *sums, double *yield_speed, void *stream) {
    if (!obs_rec || !ped_out || !car_out || !sums || !yield_speed) return api_fail(MHPPO_EINVAL, "null argument");
    if (E < 1 || T < 2 || n_cars < 1 || n_ped < 1 || N < 1) return api_fail(MHPPO_EINVAL, "bad dimensions");
    StatsDims d; d.E = E; d.T = T; d.C = n_cars; d.P = n_ped; d.car_w = car_w; d.env_w = env_w; d.n_obs = car_w * n_cars + env_w + 9 * n_ped; d.N = N;
    StatsOut o; o.ped = ped_out; o.car = car_out; o.sums = sums; o.yield_speed = yield_speed;
    const dim3 grid((unsigned)((N + 127) / 128), (unsigned)E);
    k_episode_stats<<<grid, 128, 0, (cudaStream_t)stream>>>(d, obs_rec, dt, o);
    api_count_launch();
    return ck(cudaGetLastError(), "k_episode_stats");
}

int mhppo_set_gaussian_head(float mean, float std, float variance, float acc_hi) {
    if (!(std > 0.f) || !(variance > 0.f)) return api_fail(MHPPO_EINVAL, "std and variance must be > 0");
    g_head = make_head(mean, std, variance, acc_hi);
    return 0;
}

int mhppo_set_mlp_mode(int32_t mode) {
    if (mode < 0 || mode > 2) return api_fail(MHPPO_EINVAL, "mode must be 0 (auto), 1 (ffma) or 2 (tc)");
    g_mlp_mode = mode;
    return 0;
}

int mhppo_tc_failures(void) {      /* 1 if any tensor-core kernel timed out waiting for its MMAs (should never happen) */
    int v = 0;
    cudaMemcpy(&v, fail_flag(), sizeof(int), cudaMemcpyDeviceToHost);
    return v;
}

int64_t mhppo_update_workspace_bytes(int32_t n_in) {
    const int kp = padded_in(n_in);
    if (kp < 0) return -1;
    return (int64_t)(sizeof(float) * (size_t)kUpdateGridMax * net_params(kp) + 16 + sizeof(double) * (size_t)kUpdateGridMax * (4 + kDiagW));
}

static int make_set(SampleSet &ss, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN) {
    if (CN <= 0 || S % CN != 0) return api_fail(MHPPO_EINVAL, "S must be a multiple of CN");
    ss.x = x; ss.D = D; ss.S = S; ss.idx = idx; ss.CN = CN; ss.K = idx ? K : CN; ss.Q = (S / CN) * ss.K;
    if (ss.K < 0 || ss.K > CN) return api_fail(MHPPO_EINVAL, "bad selection count");
    return 0;
}

int mhppo_value_stats(int32_t n_in, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                      const float *critic, const float *rtg, float *V, double *stats3, void *workspace, void *stream) {
    if (!x || !critic || !rtg || !V || !stats3 || !workspace) return api_fail(MHPPO_EINVAL, "null argument");
    const int kp = padded_in(n_in);
    if (kp < 0 || D > kp) return api_fail(MHPPO_EUNSUPPORTED, "unsupported input width");
    SampleSet ss;
    { const int rc0 = make_set(ss, x, D, S, idx, K, CN); if (rc0) return rc0; }
    const Workspace w = carve(workspace, kp);
    cudaStream_t s = (cudaStream_t)stream;
    if (kp == 16 && use_tc(false)) { SET_SMEM(k_value_stats_tc, smem_tc(1)); k_value_stats_tc<<<kUpdateGrid, 128, smem_tc(1), s>>>(ss, critic, rtg, V, w.spartial, fail_flag()); }
    else if (kp == 16) { SET_SMEM(k_value_stats<16>, smem_fwd<16>(1)); k_value_stats<16><<<kUpdateGrid, kFwdBlock, smem_fwd<16>(1), s>>>(ss, critic, rtg, V, w.spartial); }
    else if (kp == 32) { SET_SMEM(k_value_stats<32>, smem_fwd<32>(1)); k_value_stats<32><<<kUpdateGrid, kFwdBlock, smem_fwd<32>(1), s>>>(ss, critic, rtg, V, w.spartial); }
    else { SET_SMEM(k_value_stats<56>, smem_fwd<56>(1)); k_value_stats<56><<<kUpdateGrid, kFwdBlock, smem_fwd<56>(1), s>>>(ss, critic, rtg, V, w.spartial); }
    api_count_launch();
    int rc = ck(cudaGetLastError(), "k_value_stats");
    if (rc) return rc;
    k_reduce_scalars<<<1, 32, 0, s>>>(w.spartial, kUpdateGrid, 3, stats3);
    api_count_launch();
    return ck(cudaGetLastError(), "k_reduce_scalars");
}

static int ppo_grad_impl(int32_t n_in, int32_t head, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                         const float *net, const float *act, const float *logp_old, const float *rtg, const float *V, float adv_mean,
                         float adv_inv_std, float inv_n, float f0, float f1, float *grad, double *loss, float *V_out, double *stats3,
                         const double *adv_stats_dev, void *workspace, void *stream, float ent_coef = 0.f,
                         double *diag_row = nullptr, float *kl_slot = nullptr) {
    if (!x || !net || !rtg || !grad || !loss || !workspace) return api_fail(MHPPO_EINVAL, "null argument");
    if (head < 0 || head > 2) return api_fail(MHPPO_EINVAL, "head must be 0, 1 or 2");
    if (head != 0 && (!act || !logp_old || !V)) return api_fail(MHPPO_EINVAL, "actor heads need act, logp_old and V");
    const int kp = padded_in(n_in);
    if (kp < 0 || D > kp) return api_fail(MHPPO_EUNSUPPORTED, "unsupported input width");
    SampleSet ss;
    { const int rc0 = make_set(ss, x, D, S, idx, K, CN); if (rc0) return rc0; }
    const Workspace w = carve(workspace, kp);
    LossArgs la; la.act = act; la.logp_old = logp_old; la.rtg = rtg; la.V = V; la.adv_mean = adv_mean; la.adv_inv_std = adv_inv_std;
    la.inv_n = inv_n; la.f0 = f0; la.f1 = f1; la.V_out = V_out; la.spartial = stats3 ? w.spartial : nullptr;
    la.head = g_head; la.stats_dev = adv_stats_dev; la.ent_coef = ent_coef; la.dpartial = w.dpartial;
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if (diag_row) rc = (kp == 16) ? launch_grad<16, true>(head, ss, net, la, w, s) : ((kp == 32) ? launch_grad<32, true>(head, ss, net, la, w, s) : launch_grad<56, true>(head, ss, net, la, w, s));
    else rc = (kp == 16) ? launch_grad<16, false>(head, ss, net, la, w, s) : ((kp == 32) ? launch_grad<32, false>(head, ss, net, la, w, s) : launch_grad<56, false>(head, ss, net, la, w, s));
    if (rc) return rc;
    const int npar = net_params(kp);
    k_reduce_all<<<(npar + 255) / 256, 256, 0, s>>>(w.gpartial, kGradGrid, npar, grad, w.lpartial, loss, w.spartial, stats3);
    api_count_launch();
    if ((rc = ck(cudaGetLastError(), "k_reduce_all")) || !diag_row) return rc;
    k_reduce_diag<<<1, 32, 0, s>>>(w.lpartial, w.dpartial, kGradGrid, head, diag_row, kl_slot);
    api_count_launch();
    return ck(cudaGetLastError(), "k_reduce_diag");
}

int mhppo_ppo_grad(int32_t n_in, int32_t head, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                   const float *net, const float *act, const float *logp_old, const float *rtg, const float *V, float adv_mean,
                   float adv_inv_std, float inv_n, float f0, float f1, float *grad, double *loss, void *workspace, void *stream) {
    return ppo_grad_impl(n_in, head, x, D, S, idx, K, CN, net, act, logp_old, rtg, V, adv_mean, adv_inv_std, inv_n, f0, f1, grad, loss,
                         nullptr, nullptr, nullptr, workspace, stream);
}

int mhppo_ppo_grad_dev(int32_t n_in, int32_t head, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                       const float *net, const float *act, const float *logp_old, const float *rtg, const float *V,
                       const double *adv_stats_dev, float inv_n, float f0, float f1, float *grad, double *loss, void *workspace,
                       void *stream) {
    if (!adv_stats_dev) return api_fail(MHPPO_EINVAL, "null argument");
    return ppo_grad_impl(n_in, head, x, D, S, idx, K, CN, net, act, logp_old, rtg, V, 0.f, 0.f, inv_n, f0, f1, grad, loss, nullptr, nullptr,
                         adv_stats_dev, workspace, stream);
}

int mhppo_ppo_grad_ent(int32_t n_in, int32_t head, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                       const float *net, const float *act, const float *logp_old, const float *rtg, const float *V,
                       const double *adv_stats_dev, float inv_n, float f0, float f1, float ent_coef, float *grad, double *loss,
                       void *workspace, void *stream) {
    if (!adv_stats_dev) return api_fail(MHPPO_EINVAL, "null argument");
    if (!std::isfinite(ent_coef)) return api_fail(MHPPO_EINVAL, "ent_coef must be finite");
    if (ent_coef != 0.f && head != 2) return api_fail(MHPPO_EINVAL, "the entropy bonus needs head 2 (categorical choice actor)");
    return ppo_grad_impl(n_in, head, x, D, S, idx, K, CN, net, act, logp_old, rtg, V, 0.f, 0.f, inv_n, f0, f1, grad, loss, nullptr, nullptr,
                         adv_stats_dev, workspace, stream, ent_coef);
}

int mhppo_critic_grad_diag(int32_t n_in, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                           const float *critic, const float *rtg, float inv_n, float *grad, double *loss, float *V, double *stats3,
                           double *record_row, void *workspace, void *stream) {
    if (!record_row) return api_fail(MHPPO_EINVAL, "null argument");
    if (!V != !stats3) return api_fail(MHPPO_EINVAL, "V and stats3 go together (both null: the critic pass of GAE mode)");
    return ppo_grad_impl(n_in, 0, x, D, S, idx, K, CN, critic, nullptr, nullptr, rtg, nullptr, 0.f, 0.f, inv_n, 0.f, 0.f, grad, loss, V,
                         stats3, nullptr, workspace, stream, 0.f, record_row, nullptr);
}

int mhppo_ppo_grad_diag(int32_t n_in, int32_t head, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                        const float *net, const float *act, const float *logp_old, const float *rtg, const float *V,
                        const double *adv_stats_dev, float inv_n, float f0, float f1, float ent_coef, float *grad, double *loss,
                        float *kl_slot, double *record_row, void *workspace, void *stream) {
    if (!adv_stats_dev || !record_row) return api_fail(MHPPO_EINVAL, "null argument");
    if (head != 1 && head != 2) return api_fail(MHPPO_EINVAL, "head must be 1 or 2 (the critic pass is mhppo_critic_grad_diag)");
    if (!std::isfinite(ent_coef)) return api_fail(MHPPO_EINVAL, "ent_coef must be finite");
    if (ent_coef != 0.f && head != 2) return api_fail(MHPPO_EINVAL, "the entropy bonus needs head 2 (categorical choice actor)");
    return ppo_grad_impl(n_in, head, x, D, S, idx, K, CN, net, act, logp_old, rtg, V, 0.f, 0.f, inv_n, f0, f1, grad, loss, nullptr, nullptr,
                         adv_stats_dev, workspace, stream, ent_coef, record_row, kl_slot);
}

int mhppo_gae(const float *rew, const float *V, const int8_t *route, int32_t T, int64_t CN, double gamma, double lambda, float *ret,
              double *stats6, void *workspace, void *stream) {
    if (!rew || !V || !route || !ret || !stats6 || !workspace) return api_fail(MHPPO_EINVAL, "null argument");
    if (T < 1 || CN < 1) return api_fail(MHPPO_EINVAL, "T and CN must be >= 1");
    if (!(gamma >= 0.0 && gamma <= 1.0) || !(lambda >= 0.0 && lambda <= 1.0)) return api_fail(MHPPO_EINVAL, "gamma and lambda must lie in [0, 1]");
    const int64_t blocks = (CN + kGaeBlock - 1) / kGaeBlock;
    const int cap = 8 * sm_count() < kGaeGridMax ? 8 * sm_count() : kGaeGridMax;
    const int grid = blocks < cap ? (int)blocks : cap;
    double *partial = (double *)workspace;
    cudaStream_t s = (cudaStream_t)stream;
    k_gae<<<grid, kGaeBlock, 0, s>>>(rew, V, route, T, CN, gamma, lambda, ret, partial);
    api_count_launch();
    int rc = ck(cudaGetLastError(), "k_gae");
    if (rc) return rc;
    k_reduce_gae<<<1, 192, 0, s>>>(partial, grid, stats6);
    api_count_launch();
    return ck(cudaGetLastError(), "k_reduce_gae");
}

int mhppo_minibatch_plan(const mhppo_rollout_cfg *cfg, const int8_t *route, const int8_t *exist, const float *act_d, uint32_t iteration,
                         int32_t epochs, int32_t n_minibatches, int32_t *lists, int64_t *offsets, int64_t *counts, void *workspace,
                         void *stream) {
    if (!cfg || !route || !exist || !act_d || !lists || !offsets || !counts || !workspace) return api_fail(MHPPO_EINVAL, "null argument");
    if (epochs < 1) return api_fail(MHPPO_EINVAL, "epochs must be >= 1");
    if (n_minibatches < 1 || n_minibatches > kMbMaxBuckets) return api_fail(MHPPO_EINVAL, "n_minibatches must lie in [1, 1024]");
    const RolloutDims d = dims_of(cfg);
    const int64_t M = (int64_t)d.C * d.N;
    if (d.N < 1 || d.C < 1 || M > 0x7fffffff) return api_fail(MHPPO_EINVAL, "bad rollout dimensions");
    MbPlanArgs a;
    a.d = d; a.route = route; a.exist = exist; a.act_d = act_d; a.iteration = iteration; a.E = epochs; a.B = n_minibatches; a.M = M;
    const int64_t per = (M + kMbMaxTiles - 1) / kMbMaxTiles;
    a.tile = (per + kMbBlock - 1) / kMbBlock * kMbBlock;
    a.tiles = (int)((M + a.tile - 1) / a.tile);
    a.hist = (int32_t *)workspace; a.lists = lists; a.offsets = offsets; a.counts = counts;
    cudaStream_t s = (cudaStream_t)stream;
    k_mb_count<<<dim3((unsigned)a.tiles, (unsigned)epochs), kMbBlock, 0, s>>>(a);
    api_count_launch();
    int rc = ck(cudaGetLastError(), "k_mb_count");
    if (rc) return rc;
    k_mb_scan<<<dim3((unsigned)epochs, kMbRows), kMbMaxBuckets, 0, s>>>(a);
    api_count_launch();
    if ((rc = ck(cudaGetLastError(), "k_mb_scan"))) return rc;
    k_mb_scatter<<<dim3((unsigned)a.tiles, (unsigned)epochs), kMbBlock, 0, s>>>(a);
    api_count_launch();
    return ck(cudaGetLastError(), "k_mb_scatter");
}

int mhppo_critic_grad_stats(int32_t n_in, const float *x, int32_t D, int64_t S, const int32_t *idx, int64_t K, int64_t CN,
                            const float *critic, const float *rtg, float inv_n, float *grad, double *loss, float *V, double *stats3,
                            void *workspace, void *stream) {
    if (!V || !stats3) return api_fail(MHPPO_EINVAL, "null argument");
    return ppo_grad_impl(n_in, 0, x, D, S, idx, K, CN, critic, nullptr, nullptr, rtg, nullptr, 0.f, 0.f, inv_n, 0.f, 0.f, grad, loss, V,
                         stats3, nullptr, workspace, stream);
}

int mhppo_adam(float *p, const float *g, float *m, float *v, int32_t n, float lr, float beta1, float beta2, float eps, int32_t step,
               float grad_scale, void *stream) {
    if (!p || !g || !m || !v || n <= 0 || step < 1) return api_fail(MHPPO_EINVAL, "bad argument");
    const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
    k_adam<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, beta1, beta2, step_size, inv_sqrt_bc2, eps, grad_scale);
    api_count_launch();
    return ck(cudaGetLastError(), "k_adam");
}

int mhppo_adam2(float *p0, const float *g0, float *m0, float *v0, int32_t n0, float lr0, int32_t step0, float *p1, const float *g1,
                float *m1, float *v1, int32_t n1, float lr1, int32_t step1, float beta1, float beta2, float eps, void *stream) {
    if (!p0 || !g0 || !m0 || !v0 || !p1 || !g1 || !m1 || !v1 || n0 <= 0 || n1 <= 0 || step0 < 1 || step1 < 1) return api_fail(MHPPO_EINVAL, "bad argument");
    auto mk = [&](float *p, const float *g, float *m, float *v, int n, float lr, int step) {
        const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
        AdamArgs a; a.p = p; a.g = g; a.m = m; a.v = v; a.n = n; a.step_size = (float)((double)lr / bc1); a.inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
        return a;
    };
    const int nmax = n0 > n1 ? n0 : n1;
    k_adam2<<<dim3((nmax + 255) / 256, 2), 256, 0, (cudaStream_t)stream>>>(mk(p0, g0, m0, v0, n0, lr0, step0), mk(p1, g1, m1, v1, n1, lr1, step1), beta1, beta2, eps);
    api_count_launch();
    return ck(cudaGetLastError(), "k_adam2");
}

int mhppo_adam2_halt(float *p0, const float *g0, float *m0, float *v0, int32_t n0, float lr0, int32_t step0, float *p1, const float *g1,
                     float *m1, float *v1, int32_t n1, float lr1, int32_t step1, float beta1, float beta2, float eps,
                     const float *kl_sum, double kl_limit, int32_t *halt, double *record_row, void *stream) {
    if (!p0 || !g0 || !m0 || !v0 || !p1 || !g1 || !m1 || !v1 || n0 <= 0 || n1 <= 0 || step0 < 1 || step1 < 1) return api_fail(MHPPO_EINVAL, "bad argument");
    if (!kl_sum || !halt || !record_row) return api_fail(MHPPO_EINVAL, "null argument");
    if (std::isnan(kl_limit)) return api_fail(MHPPO_EINVAL, "kl_limit must not be NaN");
    auto mk = [&](float *p, const float *g, float *m, float *v, int n, float lr, int step) {
        const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
        AdamArgs a; a.p = p; a.g = g; a.m = m; a.v = v; a.n = n; a.step_size = (float)((double)lr / bc1); a.inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
        return a;
    };
    const int nmax = n0 > n1 ? n0 : n1;
    k_adam2_halt<<<dim3((nmax + 255) / 256, 2), 256, 0, (cudaStream_t)stream>>>(mk(p0, g0, m0, v0, n0, lr0, step0), mk(p1, g1, m1, v1, n1, lr1, step1),
                                                                               beta1, beta2, eps, kl_sum, kl_limit, (int *)halt, record_row + 9);
    api_count_launch();
    return ck(cudaGetLastError(), "k_adam2_halt");
}

int mhppo_adam2_clip(float *p0, const float *g0, float *m0, float *v0, int32_t n0, float lr0, int32_t step0, float *p1, const float *g1,
                     float *m1, float *v1, int32_t n1, float lr1, int32_t step1, float beta1, float beta2, float eps, double max_norm,
                     double *norms_out, const float *kl_sum, double kl_limit, int32_t *halt, double *record_row, void *stream) {
    if (!p0 || !g0 || !m0 || !v0 || !p1 || !g1 || !m1 || !v1 || n0 <= 0 || n1 <= 0 || step0 < 1 || step1 < 1) return api_fail(MHPPO_EINVAL, "bad argument");
    if (!(max_norm > 0.0)) return api_fail(MHPPO_EINVAL, "max_norm must be > 0 (+inf records the norms without clipping)");
    const int nhalt = (kl_sum != nullptr) + (halt != nullptr) + (record_row != nullptr);
    if (nhalt != 0 && nhalt != 3) return api_fail(MHPPO_EINVAL, "kl_sum, halt and record_row go together (all null: no halt)");
    if (nhalt && std::isnan(kl_limit)) return api_fail(MHPPO_EINVAL, "kl_limit must not be NaN");
    auto mk = [&](float *p, const float *g, float *m, float *v, int n, float lr, int step) {
        const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
        AdamArgs a; a.p = p; a.g = g; a.m = m; a.v = v; a.n = n; a.step_size = (float)((double)lr / bc1); a.inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
        return a;
    };
    const AdamArgs a0 = mk(p0, g0, m0, v0, n0, lr0, step0), a1 = mk(p1, g1, m1, v1, n1, lr1, step1);
    if (nhalt)
        k_adam2_clip<true><<<dim3(1, 2), kClipBlock, 0, (cudaStream_t)stream>>>(a0, a1, beta1, beta2, eps, max_norm, norms_out, kl_sum, kl_limit,
                                                                                (int *)halt, record_row + 9);
    else
        k_adam2_clip<false><<<dim3(1, 2), kClipBlock, 0, (cudaStream_t)stream>>>(a0, a1, beta1, beta2, eps, max_norm, norms_out, nullptr, 0.0,
                                                                                 nullptr, nullptr);
    api_count_launch();
    return ck(cudaGetLastError(), "k_adam2_clip");
}

int mhppo_adam2_sched(float *p0, const float *g0, float *m0, float *v0, int32_t n0, float lr0, int32_t step0, float *p1, const float *g1,
                      float *m1, float *v1, int32_t n1, float lr1, int32_t step1, float beta1, float beta2, float eps, double max_norm,
                      double *norms_out, const float *kl_sum, double kl_limit, int32_t *halt, double *record_row, float *lr_dev,
                      const float *kl_sum_dev, double n, double desired_kl, double *lrs_out_dev, void *stream) {
    if (!p0 || !g0 || !m0 || !v0 || !p1 || !g1 || !m1 || !v1 || n0 <= 0 || n1 <= 0 || step0 < 1 || step1 < 1) return api_fail(MHPPO_EINVAL, "bad argument");
    if (!(max_norm > 0.0)) return api_fail(MHPPO_EINVAL, "max_norm must be > 0 (+inf: no clipping)");
    const int nhalt = (kl_sum != nullptr) + (halt != nullptr) + (record_row != nullptr);
    if (nhalt != 0 && nhalt != 3) return api_fail(MHPPO_EINVAL, "kl_sum, halt and record_row go together (all null: no halt)");
    if (nhalt && std::isnan(kl_limit)) return api_fail(MHPPO_EINVAL, "kl_limit must not be NaN");
    if (!lr_dev || !kl_sum_dev) return api_fail(MHPPO_EINVAL, "null argument");
    if (!(desired_kl > 0.0)) return api_fail(MHPPO_EINVAL, "desired_kl must be > 0");
    if (!(n > 0.0)) return api_fail(MHPPO_EINVAL, "n must be > 0");
    auto mk = [&](float *p, const float *g, float *m, float *v, int n, float lr, int step) {
        const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
        AdamArgs a; a.p = p; a.g = g; a.m = m; a.v = v; a.n = n; a.step_size = (float)((double)lr / bc1); a.inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
        return a;
    };
    AdaptArgs ad;
    ad.lr = lr_dev; ad.kl_sum = kl_sum_dev; ad.lrs_out = lrs_out_dev; ad.n = n; ad.desired_kl = desired_kl;
    ad.bc1[0] = 1.0 - std::pow((double)beta1, (double)step0);
    ad.bc1[1] = 1.0 - std::pow((double)beta1, (double)step1);
    const AdamArgs a0 = mk(p0, g0, m0, v0, n0, lr0, step0), a1 = mk(p1, g1, m1, v1, n1, lr1, step1);
    if (nhalt)
        k_adam2_clip<true, true><<<dim3(1, 2), kClipBlock, 0, (cudaStream_t)stream>>>(a0, a1, beta1, beta2, eps, max_norm, norms_out, kl_sum,
                                                                                      kl_limit, (int *)halt, record_row + 9, ad);
    else
        k_adam2_clip<false, true><<<dim3(1, 2), kClipBlock, 0, (cudaStream_t)stream>>>(a0, a1, beta1, beta2, eps, max_norm, norms_out,
                                                                                       nullptr, 0.0, nullptr, nullptr, ad);
    api_count_launch();
    return ck(cudaGetLastError(), "k_adam2_clip");
}

}  // extern "C"
