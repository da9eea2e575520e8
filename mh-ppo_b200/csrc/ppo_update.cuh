// ppo_update.cuh -- update-side kernels of the PPO loop (Algo_PPO.train_model_c / train_model_d,
// PY:778-851): critic forward + advantage statistics, fused actor/critic forward + clipped-surrogate
// / MSE loss + backward with per-CTA gradient accumulation, deterministic gradient reduction, Adam.
//
// One epoch of train_model_c over the samples selected by `route` (cross or wait buffer):
//   1. k_value_stats : V = critic(s), A = RTG - V, per-CTA partial (sum A, sum A^2, n) in fp64
//   2. (host: reduce partials; multi-GPU: all-reduce the 3 scalars -> global mean / unbiased std)
//   3. k_ppo_grad    : forward both nets, loss epilogue, backward, dW partial per CTA
//   4. k_reduce      : fixed-order sum of the CTA partials -> flat gradient (deterministic)
//   5. (multi-GPU: one NCCL all-reduce of the flat gradient buffer)       6. k_adam
//
// Execution model: thread = sample(s) for forward and backward-data (activations of the CTA's tile sit
// in shared memory as [sample][feature], deltas overwrite activations in place), then the same 128
// threads switch roles and each owns a register tile of every weight matrix for the weight
// gradient dWt[k][j] += sum_s in[s][k] * delta[s][j], accumulated across all tiles of a
// persistent CTA (one per SM).
#pragma once
#include "mlp.cuh"
#include "ppo_rollout.cuh"      // policy_block: the minibatch plan draws from stream 3 of the policy-noise contract

namespace mhppo {

struct SampleSet {
    const float *x;        // features, feature-major [D][S]
    int D;                 // real feature count (<= KP)
    int64_t S;             // sample slots in the buffers (row pitch of x)
    const int32_t *idx;    // compacted list of the selected (car, env) columns m in [0, CN), or null = every column
    int64_t K;             // number of selected columns (CN when idx is null)
    int64_t CN;            // columns per time step; sample slot s = t*CN + m
    int64_t Q;             // work items = T*K; item q -> (t = q / K, k = q % K)
};
// work item -> sample slot; false past the end.  The update walks only the samples routed to the net being
// trained (cross or wait buffer, PY:489-502), so every lane of a tile is busy.
__device__ __forceinline__ bool map_sample(const SampleSet &ss, int64_t q, int64_t &s) {
    if (q >= ss.Q) return false;
    const int64_t t = q / ss.K, k = q - t * ss.K;
    s = t * ss.CN + (ss.idx ? (int64_t)ss.idx[k] : k);
    return true;
}

template <int KP>
__device__ __forceinline__ void load_row(const SampleSet &ss, int64_t s, float *x) {
#pragma unroll
    for (int k = 0; k < KP; ++k) x[k] = (k < ss.D) ? ss.x[(int64_t)k * ss.S + s] : 0.f;
}

// sum over a team of `nthreads` consecutive threads (a whole CTA, or one 128-thread team of it synchronising on its own
// named barrier `bar`); the result is valid in the team's first thread
__device__ __forceinline__ void team_sync(int bar, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(nthreads) : "memory"); }
__device__ __forceinline__ double team_sum(double v, double *red, int ltid, int nthreads, int bar) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((ltid & 31) == 0) red[ltid >> 5] = v;
    team_sync(bar, nthreads);
    double r = 0.0;
    if (ltid == 0) for (int w = 0; w < nthreads / 32; ++w) r += red[w];
    team_sync(bar, nthreads);
    return r;
}

// ---- 1. critic forward + advantage statistics --------------------------------------------------------
template <int KP>
__global__ void __launch_bounds__(kFwdBlock, 2) k_value_stats(SampleSet ss, const float *__restrict__ critic, const float *__restrict__ rtg,
                                                           float *__restrict__ V, double *__restrict__ partial /* [grid][3] */) {
    extern __shared__ __align__(16) float smem[];
    float *sw = smem;
    float *rows = smem + ((net_params(KP) + 3) & ~3);
    __shared__ double red[kFwdBlock / 32];
    stage_net<KP>(sw, critic);
    __syncthreads();
    float *x = rows + (size_t)threadIdx.x * kRowFwd;      // one in-place row per sample
    double sA = 0.0, sAA = 0.0, cnt = 0.0;
    for (int64_t base = (int64_t)blockIdx.x * kFwdBlock; base < ss.Q; base += (int64_t)gridDim.x * kFwdBlock) {
        int64_t s = 0;
        if (map_sample(ss, base + threadIdx.x, s)) {
            load_row<KP>(ss, s, x);
            const float v = mlp_fwd_inplace<KP>(sw, x).x;
            V[s] = v;
            const double A = (double)(rtg[s] - v);          // advantage_batch = rtgs - V, fp32 like torch (PY:786)
            sA += A; sAA += A * A; cnt += 1.0;
        }
    }
    const double t0 = team_sum(sA, red, threadIdx.x, kFwdBlock, 0), t1 = team_sum(sAA, red, threadIdx.x, kFwdBlock, 0),
                 t2 = team_sum(cnt, red, threadIdx.x, kFwdBlock, 0);
    if (threadIdx.x == 0) { partial[blockIdx.x * 3 + 0] = t0; partial[blockIdx.x * 3 + 1] = t1; partial[blockIdx.x * 3 + 2] = t2; }
}

// ---- 3. fused forward + loss + backward ----------------------------------------------------------------
struct LossArgs {
    const float *act, *logp_old, *rtg, *V;     // per-sample
    float adv_mean, adv_inv_std;               // (A - mean) * inv_std, inv_std = 1 / (std_unbiased + 1e-10)  (PY:787)
    float inv_n;                               // 1 / (global sample count)
    float f0, f1;                              // choice only: fraction of samples whose action is 0 / 1 (PY:834-842 broadcast)
    float *V_out;                              // critic only, optional: V[s] of this forward pass and the advantage statistics
    double *spartial;                          //   [grid][3] partial (sum A, sum A^2, n) with A = rtg - V (replaces k_value_stats)
    HeadCfg head;                              // Gaussian head (HEAD == 1)
    const double *stats_dev;                   // actor heads, optional: (sum A, sum A^2, n) of the whole (all-rank) batch in device
                                               //   memory; adv_mean / adv_inv_std are then derived in the kernel (no host round trip)
    float ent_coef;                            // choice only: entropy bonus c; read only by the k_ppo_grad<KP, 2, true> instances
    double *dpartial;                          // DIAG instances only: [grid][kDiagW] per-CTA diagnostic sums (LossAcc)
};

// advantage normalisation of PY:787 from the partial sums: mean, 1 / (unbiased std + 1e-10) (Algo_PPO.combine_stats)
__device__ __forceinline__ void resolve_adv_stats(LossArgs &la) {
    if (!la.stats_dev) return;
    const double sA = la.stats_dev[0], sAA = la.stats_dev[1], n = la.stats_dev[2];
    if (n < 1.0) { la.adv_mean = 0.f; la.adv_inv_std = 0.f; return; }
    const double mean = sA / n;
    const double var = (n > 1.0) ? fmax(sAA - n * mean * mean, 0.0) / (n - 1.0) : nan("");
    la.adv_mean = (float)mean; la.adv_inv_std = (float)(1.0 / (sqrt(var) + 1e-10));
}

// ---- register-tiled dense layers for the fused kernel -------------------------------------------------
// The first version read one weight per FFMA from shared memory (a 128-bit broadcast load feeds 4 FFMAs of
// one sample) and the weight-gradient strips read one delta per FFMA: 3 shared-memory wavefront cycles per
// FFMA issue cycle, FMA pipe 27 % busy (profiles/round1_ppo_kernels_summary.txt).  Here every thread owns R
// samples (rows tid, tid + 128, ...) so a weight load feeds R x 4 FFMAs, every row access is a 128-bit
// load/store (rows are 16-byte aligned, row stride = 4 mod 32 words: 8 lanes x 16 B per wavefront, conflict-free),
// and the weight gradient is a 4 x 8 register tile per thread.
template <int KP>
struct GradCfg {
    static constexpr int R = (KP <= 16) ? 2 : 1;                    // samples per thread (shared memory bounds it)
    static constexpr int TILE = kMlpBlock * R;                      // samples per CTA tile
    static constexpr int X = 0, A1 = KP, A2 = KP + H1, A3 = KP + H1 + H2, D4 = KP + H1 + H2 + H3, RAW = D4 + OP;
    static constexpr int ROW = ((RAW - 4 + 31) / 32) * 32 + 4;      // >= RAW and = 4 (mod 32)
    static constexpr int NPAR = net_params(KP), NP4 = (NPAR + 3) & ~3;
    static constexpr size_t smem_floats = (size_t)NP4 + H2 * H1 + H3 * H2 + OP * H3 + (size_t)TILE * ROW;
};

__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void st4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }

// out[r][j] = act(b[j] + sum_k in[r][k] * Wt[k][j]) for the R rows of this thread; rows are `rs` floats apart
template <int K, int J, bool RELU, int R>
__device__ __forceinline__ void dense_fwd_t(const float *in, float *out, int rs, const float *__restrict__ Wt, const float *__restrict__ b) {
    constexpr int JC = (J < 32) ? J : 32;
#pragma unroll 1
    for (int jc = 0; jc < J; jc += JC) {
        float acc[R][JC];
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int j = 0; j < JC; ++j) acc[r][j] = b[jc + j];
#pragma unroll 2
        for (int k = 0; k < K; k += 4) {
            float a[R][4];
#pragma unroll
            for (int r = 0; r < R; ++r) { const float4 v = ld4(in + r * rs + k); a[r][0] = v.x; a[r][1] = v.y; a[r][2] = v.z; a[r][3] = v.w; }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                for (int j4 = 0; j4 < JC / 4; ++j4) {
                    const float4 w = ld4(Wt + (k + kk) * J + jc + 4 * j4);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        acc[r][4 * j4 + 0] = fmaf(a[r][kk], w.x, acc[r][4 * j4 + 0]); acc[r][4 * j4 + 1] = fmaf(a[r][kk], w.y, acc[r][4 * j4 + 1]);
                        acc[r][4 * j4 + 2] = fmaf(a[r][kk], w.z, acc[r][4 * j4 + 2]); acc[r][4 * j4 + 3] = fmaf(a[r][kk], w.w, acc[r][4 * j4 + 3]);
                    }
                }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int j4 = 0; j4 < JC / 4; ++j4) {
                float4 o = make_float4(acc[r][4 * j4], acc[r][4 * j4 + 1], acc[r][4 * j4 + 2], acc[r][4 * j4 + 3]);
                if (RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                st4(out + r * rs + jc + 4 * j4, o);
            }
    }
}

// backward-data for the R rows of this thread: din[k] = relu'(ain[k]) * sum_j dout[j] * W[j][k], written over ain
template <int K, int J, int R>
__device__ __forceinline__ void dense_bwd_t(float *ain_din, const float *dout, int rs, const float *__restrict__ W /* [J][K] */) {
    constexpr int KC = (K < 32) ? K : 32;
#pragma unroll 1
    for (int kc = 0; kc < K; kc += KC) {
        float acc[R][KC];
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int k = 0; k < KC; ++k) acc[r][k] = 0.f;
#pragma unroll 2
        for (int j = 0; j < J; j += 4) {
            float d[R][4];
#pragma unroll
            for (int r = 0; r < R; ++r) { const float4 v = ld4(dout + r * rs + j); d[r][0] = v.x; d[r][1] = v.y; d[r][2] = v.z; d[r][3] = v.w; }
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                for (int k4 = 0; k4 < KC / 4; ++k4) {
                    const float4 w = ld4(W + (j + jj) * K + kc + 4 * k4);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        acc[r][4 * k4 + 0] = fmaf(d[r][jj], w.x, acc[r][4 * k4 + 0]); acc[r][4 * k4 + 1] = fmaf(d[r][jj], w.y, acc[r][4 * k4 + 1]);
                        acc[r][4 * k4 + 2] = fmaf(d[r][jj], w.z, acc[r][4 * k4 + 2]); acc[r][4 * k4 + 3] = fmaf(d[r][jj], w.w, acc[r][4 * k4 + 3]);
                    }
                }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int k4 = 0; k4 < KC / 4; ++k4) {
                float *q = ain_din + r * rs + kc + 4 * k4;
                const float4 av = ld4(q);
                st4(q, make_float4(av.x > 0.f ? acc[r][4 * k4] : 0.f, av.y > 0.f ? acc[r][4 * k4 + 1] : 0.f,
                                   av.z > 0.f ? acc[r][4 * k4 + 2] : 0.f, av.w > 0.f ? acc[r][4 * k4 + 3] : 0.f));
            }
    }
}

#ifndef MH_WGRAD_UNROLL_N
#define MH_WGRAD_UNROLL_N 2
#endif
constexpr int MH_WGRAD_UNROLL = MH_WGRAD_UNROLL_N;      // rows in flight per thread in the weight-gradient loops
// weight-gradient register tile: acc[kk][j] += in[s][k0 + kk] * delta[s][j0 + j] over the rows [s0, s0 + ns) of the tile
template <int TJ>
__device__ __forceinline__ void wgrad_tile(float (&acc)[4][TJ], const float *__restrict__ rows, int row, int in_off, int dl_off, int s0, int ns) {
#pragma unroll 2
    for (int s = s0; s < s0 + ns; ++s) {
        const float *r = rows + (size_t)s * row;
        const float4 av = ld4(r + in_off);
        const float a[4] = {av.x, av.y, av.z, av.w};
        float d[TJ];
        if (TJ == 2) { const float2 v = *reinterpret_cast<const float2 *>(r + dl_off); d[0] = v.x; d[1] = v.y; }
        else {
#pragma unroll
            for (int j4 = 0; j4 < TJ / 4; ++j4) { const float4 v = ld4(r + dl_off + 4 * j4); d[4 * j4] = v.x; d[4 * j4 + 1] = v.y; d[4 * j4 + 2] = v.z; d[4 * j4 + 3] = v.w; }
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
#pragma unroll
            for (int j = 0; j < TJ; ++j) acc[kk][j] = fmaf(a[kk], d[j], acc[kk][j]);
    }
}

// ---- loss epilogue of one sample (shared by the FFMA and the tensor-core kernel) ------------------------
// HEAD: 0 = critic (MSE), 1 = Gaussian actor (clipped surrogate), 2 = categorical actor with the (M,M) broadcast.
// o: raw outputs of the net; returns dLoss/dz (4 padded outputs) and accumulates the loss and, for the critic,
// the advantage statistics.
// The DIAG instances also sum, per thread in fp64, the update diagnostics (DESIGN.md §4 "Diagnostics"): for the actor heads the
// k3 estimator r - 1 - log r, the clipped-ratio count and (choice) the entropy; for the critic R - V, (R - V)^2, R and R^2.
constexpr int kDiagW = 4;                  // diagnostic partials per CTA: actor (k3, clipped, H, 0), critic (R-V, (R-V)^2, R, R^2)
struct LossAcc {
    double loss = 0.0, sA = 0.0, sAA = 0.0, cnt = 0.0;
    double d[kDiagW] = {0.0, 0.0, 0.0, 0.0};
};
// the per-sample inputs of the loss (rtg for every head; V, action, old log-prob for the actors): can be loaded ahead of use
struct LossIn { float rtg, V, act, logp; };
// (DIAG: the choice head also reads its taken action, for the per-sample ratio of the diagnostics)
template <int HEAD, bool DIAG = false>
__device__ __forceinline__ LossIn load_loss_in(const LossArgs &la, int64_t s) {
    LossIn in; in.rtg = la.rtg[s]; in.V = 0.f; in.act = 0.f; in.logp = 0.f;
    if (HEAD != 0) { in.V = la.V[s]; in.logp = la.logp_old[s]; }
    if (HEAD == 1 || (DIAG && HEAD == 2)) in.act = la.act[s];
    return in;
}
// k3 = r - 1 - log r of an fp32 log-ratio, in fp64 as expm1(l) - l: no cancellation near r = 1, finite for |l| up to ~700
__device__ __forceinline__ double k3_of(float l) { const double d = (double)l; return expm1(d) - d; }
// ENT (HEAD == 2 only): adds the entropy bonus -c * inv_n * H(pi(.|s)) to the loss; ENT = false is the reference's loss.
// DIAG: also accumulates the diagnostics of the sample into acc.d (read-only side computations: dz and acc.loss are unchanged)
template <int HEAD, bool ENT = false, bool DIAG = false>
__device__ __forceinline__ void ppo_loss(const LossArgs &la, int64_t s, const LossIn &in, float4 o, float (&dz)[OP], LossAcc &acc) {
    static_assert(!ENT || HEAD == 2, "the entropy bonus exists for the categorical head only");
    if (HEAD == 0) {                                           // critic_loss = MSE(V, rtg), PY:808-809
        const float e = o.x - in.rtg;
        acc.loss += (double)e * (double)e * (double)la.inv_n;
        dz[0] = 2.0f * e * la.inv_n;
        if (la.V_out) {                                        // V = critic(s), A = rtgs - V (PY:785-786)
            la.V_out[s] = o.x;
            const double A = (double)(in.rtg - o.x);
            acc.sA += A; acc.sAA += A * A; acc.cnt += 1.0;
        }
        if (DIAG) {                                            // explained variance: R = this pass's target, V = its forward output
            const double R = (double)in.rtg, d = R - (double)o.x;
            acc.d[0] += d; acc.d[1] += d * d; acc.d[2] += R; acc.d[3] += R * R;
        }
        return;
    }
    const float An = ((in.rtg - in.V) - la.adv_mean) * la.adv_inv_std;     // PY:786-787
    if (HEAD == 1) {
        const float th = tanhf(o.x), mu = th * la.head.std + la.head.mean;
        const float a = in.act;
        const float lp = -((a - mu) * (a - mu)) * la.head.inv_2var - la.head.logp_c;   // MVN(mu, var I).log_prob, PY:795-800
        const float ratio = expf(lp - in.logp);                           // PY:803
        const float s1 = ratio * An, s2 = fminf(fmaxf(ratio, 0.8f), 1.2f) * An;   // PY:804-805
        acc.loss += (double)(-fminf(s1, s2)) * (double)la.inv_n;                 // PY:806
        if (s1 <= s2) dz[0] = -la.inv_n * An * ratio * (2.0f * la.head.inv_2var * (a - mu)) * (la.head.std * (1.0f - th * th));
        if (DIAG) { acc.d[0] += k3_of(lp - in.logp); acc.d[1] += (ratio < 0.8f || ratio > 1.2f) ? 1.0 : 0.0; }
    } else {
        // Categorical(probs [M,2]).log_prob(actions [M,1]) broadcasts to (M,M): lp[i,j] = log p_j(a_i)
        // (PY:834-842).  With two actions the mean over i collapses to the action frequencies f0, f1.
        const float m = fmaxf(o.x, o.y), e0 = expf(o.x - m), e1 = expf(o.y - m);
        const float p0 = e0 / (e0 + e1), p1 = e1 / (e0 + e1);
        const float inv_old = expf(-in.logp);
        float dp0 = 0.f, dp1 = 0.f;
        {
            const float rr = p0 * inv_old, s1 = rr * An, s2 = fminf(fmaxf(rr, 0.8f), 1.2f) * An;
            acc.loss += (double)(-fminf(s1, s2)) * (double)(la.f0 * la.inv_n);
            if (s1 <= s2) dp0 = -la.inv_n * la.f0 * An * inv_old;
        }
        {
            const float rr = p1 * inv_old, s1 = rr * An, s2 = fminf(fmaxf(rr, 0.8f), 1.2f) * An;
            acc.loss += (double)(-fminf(s1, s2)) * (double)(la.f1 * la.inv_n);
            if (s1 <= s2) dp1 = -la.inv_n * la.f1 * An * inv_old;
        }
        // softmax backward: dz_a = p_a * (dp_a - sum_b p_b dp_b)
        const float dot = p0 * dp0 + p1 * dp1;
        dz[0] = p0 * (dp0 - dot); dz[1] = p1 * (dp1 - dot);
        if (ENT) {
            // H = -sum_k p_k log p_k with log p_k = z_k - m - log(e0 + e1): finite for logits any distance apart (p_k = 0 has
            // log p_k = z_k - m, so p_k log p_k = 0); dLoss/dz_k = c * inv_n * p_k * (log p_k + H)
            const float lse = logf(e0 + e1), lp0 = (o.x - m) - lse, lp1 = (o.y - m) - lse;
            const float H = -(p0 * lp0 + p1 * lp1), ci = la.ent_coef * la.inv_n;
            acc.loss -= (double)la.ent_coef * (double)la.inv_n * (double)H;
            dz[0] += ci * p0 * (lp0 + H); dz[1] += ci * p1 * (lp1 + H);
        }
        if (DIAG) {
            // the standard per-sample ratio of the taken action a_s (not the (M, M) broadcast the loss optimises): log r from the
            // log-softmax, the clip test on the fp32 ratio p_a * exp(-logp_old) that the loss's clamp sees, H as in the ENT term
            const float lse = logf(e0 + e1), lp0 = (o.x - m) - lse, lp1 = (o.y - m) - lse;
            const bool a1 = in.act != 0.f;
            const float rr = (a1 ? p1 : p0) * inv_old;
            acc.d[0] += k3_of((a1 ? lp1 : lp0) - in.logp);
            acc.d[1] += (rr < 0.8f || rr > 1.2f) ? 1.0 : 0.0;
            acc.d[2] += (double)(-(p0 * lp0 + p1 * lp1));
        }
    }
}

// the CTA's diagnostic sums (team of nthreads) -> dpartial[blockIdx.x][0 .. kDiagW)
__device__ __forceinline__ void write_diag_partials(const LossAcc &acc, double *__restrict__ dpartial, double *red, int tid, int nthreads) {
#pragma unroll
    for (int j = 0; j < kDiagW; ++j) {
        const double t = team_sum(acc.d[j], red, tid, nthreads, 0);
        if (tid == 0) dpartial[(size_t)blockIdx.x * kDiagW + j] = t;
    }
}

// ---- the weight-gradient register tiles of one thread (persist over all tiles of a CTA) ------------------
// The CTA's threads split into NG groups of 64; each group sums over 1/NG of the tile's rows and every thread of a
// group owns a 4 x TJ tile of every matrix; the groups are added once, after the last tile (finish).  `half` = group.
// Row layout: [x KP | a1/delta1 32 | a2/delta2 64 | a3/delta3 32 | dz 4], `row` floats apart.
template <int KP, int NG = 2>
struct WgradAcc {
    static constexpr int NKG1 = KP / 4;                                        // k-groups of layer 1
    static constexpr int JG1 = (NKG1 <= 4) ? 16 : ((NKG1 <= 8) ? 8 : 4);       // j-groups of layer 1 (NKG1 * JG1 <= 64 threads)
    static constexpr int TJ1 = H1 / JG1;
    static constexpr int X = 0, A1 = KP, A2 = KP + H1, A3 = KP + H1 + H2, D4 = KP + H1 + H2 + H3;
    float g1[4][TJ1], g2[4][8], g3[4][8], g4[2], gb4[2], gbias[2];
    int half, lt, k1, j1, k2, j2, k3, j3, k4, j4;
    bool l1_on;
    __device__ __forceinline__ void init(int tid) {
        half = tid >> 6; lt = tid & 63;
        l1_on = lt < NKG1 * JG1;
        k1 = (lt % NKG1) * 4; j1 = (lt / NKG1) * TJ1;                          // dW1t[k < KP][j < 32]
        k2 = (lt & 7) * 4; j2 = (lt >> 3) * 8;                                 // dW2t[k < 32][j < 64]
        k3 = (lt & 15) * 4; j3 = (lt >> 4) * 8;                                // dW3t[k < 64][j < 32]
        k4 = lt & 31; j4 = (lt >> 5) * 2;                                      // dW4t[k < 32][j < 4]
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
            for (int j = 0; j < TJ1; ++j) g1[kk][j] = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) { g2[kk][j] = 0.f; g3[kk][j] = 0.f; }
        }
        g4[0] = g4[1] = gb4[0] = gb4[1] = gbias[0] = gbias[1] = 0.f;
    }
    // layer 4: dW4t[k][j], b4[j] from (a3, dz) of the rows [s0, s0 + ns)
    __device__ __forceinline__ void layer4(const float *__restrict__ rows, int row, int s0, int ns) {
#pragma unroll 4
        for (int s = s0; s < s0 + ns; ++s) {
            const float *r = rows + (size_t)s * row;
            const float a = r[A3 + k4];
            const float2 d = *reinterpret_cast<const float2 *>(r + D4 + j4);
            g4[0] = fmaf(a, d.x, g4[0]); g4[1] = fmaf(a, d.y, g4[1]);
            gb4[0] += d.x; gb4[1] += d.y;
        }
    }
    __device__ __forceinline__ void layer3(const float *rows, int row, int s0, int ns) { wgrad_tile<8>(g3, rows, row, A2 + k3, A3 + j3, s0, ns); }
    __device__ __forceinline__ void layer2(const float *rows, int row, int s0, int ns) { wgrad_tile<8>(g2, rows, row, A1 + k2, A2 + j2, s0, ns); }
    // layer 1 and the bias gradients b1 | b2 | b3 (the deltas sit in a1, a2, a3 of every row: 128 consecutive columns)
    __device__ __forceinline__ void layer1_and_biases(const float *__restrict__ rows, int row, int s0, int ns) {
        if (l1_on) wgrad_tile<TJ1>(g1, rows, row, X + k1, A1 + j1, s0, ns);
#pragma unroll 4
        for (int s = s0; s < s0 + ns; ++s) {
            const float2 d = *reinterpret_cast<const float2 *>(rows + (size_t)s * row + A1 + 2 * lt);
            gbias[0] += d.x; gbias[1] += d.y;
        }
    }
    __device__ __forceinline__ void emit(float *dst, bool add) const {
        if (l1_on)
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                for (int j = 0; j < TJ1; ++j) { float &q = dst[(k1 + kk) * H1 + j1 + j]; q = add ? q + g1[kk][j] : g1[kk][j]; }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float &q2 = dst[off_w2(KP) + (k2 + kk) * H2 + j2 + j]; q2 = add ? q2 + g2[kk][j] : g2[kk][j];
                float &q3 = dst[off_w3(KP) + (k3 + kk) * H3 + j3 + j]; q3 = add ? q3 + g3[kk][j] : g3[kk][j];
            }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            float &q4 = dst[off_w4(KP) + k4 * OP + j4 + j]; q4 = add ? q4 + g4[j] : g4[j];
            if (k4 == 0) { float &qb = dst[off_b4(KP) + j4 + j]; qb = add ? qb + gb4[j] : gb4[j]; }
            const int c = 2 * lt + j;                   // column of (b1 | b2 | b3)
            const int o = (c < H1) ? (off_b1(KP) + c) : ((c < H1 + H2) ? (off_b2(KP) + c - H1) : (off_b3(KP) + c - H1 - H2));
            float &qq = dst[o]; qq = add ? qq + gbias[j] : gbias[j];
        }
    }
    // add the NG groups through `scratch` (>= net_params floats of shared memory no longer in use) and write the CTA's
    // partial gradient, loss and (critic) advantage statistics; `red` holds one double per warp of the CTA
    template <int HEAD, bool DIAG = false>
    __device__ __forceinline__ void finish(float *scratch, float *__restrict__ gpartial, double *__restrict__ lpartial, const LossArgs &la,
                                           const LossAcc &acc, double *red) const {
        constexpr int NPAR = net_params(KP), NT = 64 * NG;
        const int tid = threadIdx.x;
#pragma unroll 1
        for (int g = 0; g < NG; ++g) {                  // fixed order: deterministic
            if (half == g) emit(scratch, g > 0);
            __syncthreads();
        }
        float *gp = gpartial + (size_t)blockIdx.x * NPAR;
        for (int i = tid; i < NPAR; i += NT) gp[i] = scratch[i];
        const double lt_sum = team_sum(acc.loss, red, tid, NT, 0);
        if (tid == 0) lpartial[blockIdx.x] = lt_sum;
        if (HEAD == 0 && la.spartial) {
            const double t0 = team_sum(acc.sA, red, tid, NT, 0), t1 = team_sum(acc.sAA, red, tid, NT, 0), t2 = team_sum(acc.cnt, red, tid, NT, 0);
            if (tid == 0) { la.spartial[blockIdx.x * 3 + 0] = t0; la.spartial[blockIdx.x * 3 + 1] = t1; la.spartial[blockIdx.x * 3 + 2] = t2; }
        }
        if (DIAG) write_diag_partials(acc, la.dpartial, red, tid, NT);
    }
};

// Per tile: [thread = R samples] forward + loss + dz; then, layer by layer from the top, [register tiles] weight gradient from
// (input activation, delta) and [thread = R samples] backward-data which overwrites the activation with its delta.
constexpr int kTeams = 1;
template <int KP, int HEAD, bool ENT = false, bool DIAG = false>
__global__ void __launch_bounds__(kMlpBlock, 1) k_ppo_grad(SampleSet ss, const float *__restrict__ net, LossArgs la,
                                                           float *__restrict__ gpartial /* [grid][net_params] */,
                                                           double *__restrict__ lpartial /* [grid] */) {
    resolve_adv_stats(la);
    extern __shared__ __align__(16) float smem[];
    typedef GradCfg<KP> G;
    constexpr int R = G::R, ROW = G::ROW;
    float *sw = smem;                                  // flat net (transposed weights)
    float *W2 = sw + G::NP4;                           // [H2][H1] original orientation, for backward-data
    float *W3 = W2 + H2 * H1;                          // [H3][H2]
    float *W4 = W3 + H3 * H2;                          // [OP][H3]
    float *rows = W4 + OP * H3;
    __shared__ double red[kMlpBlock / 32];
    stage_net<KP>(sw, net);
    __syncthreads();
    for (int i = threadIdx.x; i < H1 * H2; i += blockDim.x) { const int k = i / H2, j = i % H2; W2[j * H1 + k] = sw[off_w2(KP) + i]; }
    for (int i = threadIdx.x; i < H2 * H3; i += blockDim.x) { const int k = i / H3, j = i % H3; W3[j * H2 + k] = sw[off_w3(KP) + i]; }
    for (int i = threadIdx.x; i < H3 * OP; i += blockDim.x) { const int k = i / OP, j = i % OP; W4[j * H3 + k] = sw[off_w4(KP) + i]; }
    __syncthreads();

    const int tid = threadIdx.x;
    float *my = rows + (size_t)tid * ROW;              // row of this thread's first sample; the r-th is kMlpBlock rows further
    constexpr int RS = kMlpBlock * ROW;
    WgradAcc<KP> wg;
    wg.init(tid);
    constexpr int HALF = G::TILE / 2;
    const int s0 = wg.half * HALF;
    LossAcc acc;

    for (int64_t base = (int64_t)blockIdx.x * G::TILE; base < ss.Q; base += (int64_t)gridDim.x * G::TILE) {
        bool sel[R];
        int64_t sidx[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            sidx[r] = 0;
            sel[r] = map_sample(ss, base + tid + r * kMlpBlock, sidx[r]);
            float *x = my + r * RS;
#pragma unroll
            for (int k = 0; k < KP; k += 4) {
                float4 v;
                v.x = (sel[r] && k + 0 < ss.D) ? ss.x[(int64_t)(k + 0) * ss.S + sidx[r]] : 0.f;
                v.y = (sel[r] && k + 1 < ss.D) ? ss.x[(int64_t)(k + 1) * ss.S + sidx[r]] : 0.f;
                v.z = (sel[r] && k + 2 < ss.D) ? ss.x[(int64_t)(k + 2) * ss.S + sidx[r]] : 0.f;
                v.w = (sel[r] && k + 3 < ss.D) ? ss.x[(int64_t)(k + 3) * ss.S + sidx[r]] : 0.f;
                st4(x + k, v);
            }
        }
        dense_fwd_t<KP, H1, true, R>(my + G::X, my + G::A1, RS, sw, sw + off_b1(KP));
        dense_fwd_t<H1, H2, true, R>(my + G::A1, my + G::A2, RS, sw + off_w2(KP), sw + off_b2(KP));
        dense_fwd_t<H2, H3, true, R>(my + G::A2, my + G::A3, RS, sw + off_w3(KP), sw + off_b3(KP));
        dense_fwd_t<H3, OP, false, R>(my + G::A3, my + G::D4, RS, sw + off_w4(KP), sw + off_b4(KP));
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float *row = my + r * RS;
            float dz[OP] = {0.f, 0.f, 0.f, 0.f};
            if (sel[r]) ppo_loss<HEAD, ENT, DIAG>(la, sidx[r], load_loss_in<HEAD, DIAG>(la, sidx[r]), ld4(row + G::D4), dz, acc);
            // an unselected row has x = 0 but its activations are relu(bias) != 0: its dz = 0 keeps every gradient term zero
            st4(row + G::D4, make_float4(dz[0], dz[1], dz[2], dz[3]));
        }
        __syncthreads();
        wg.layer4(rows, ROW, s0, HALF);
        __syncthreads();
        dense_bwd_t<H3, OP, R>(my + G::A3, my + G::D4, RS, W4);           // a3 now holds delta3
        __syncthreads();
        wg.layer3(rows, ROW, s0, HALF);
        __syncthreads();
        dense_bwd_t<H2, H3, R>(my + G::A2, my + G::A3, RS, W3);           // a2 now holds delta2
        __syncthreads();
        wg.layer2(rows, ROW, s0, HALF);
        __syncthreads();
        dense_bwd_t<H1, H2, R>(my + G::A1, my + G::A2, RS, W2);           // a1 now holds delta1
        __syncthreads();
        wg.layer1_and_biases(rows, ROW, s0, HALF);
        __syncthreads();
    }
    wg.template finish<HEAD, DIAG>(rows, gpartial, lpartial, la, acc, red);
}

// ---- 4. deterministic reduction of the per-CTA partials ----------------------------------------------
__global__ void __launch_bounds__(256) k_reduce_partials(const float *__restrict__ gpartial, int nblocks, int npar, float *__restrict__ grad) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= npar) return;
    float acc = 0.f;
    for (int b = 0; b < nblocks; ++b) acc += gpartial[(size_t)b * npar + i];
    grad[i] = acc;
}
// gradient partials, loss partials and (optionally) the advantage-statistics partials of one ppo_grad launch in ONE kernel
__global__ void __launch_bounds__(256) k_reduce_all(const float *__restrict__ gpartial, int nblocks, int npar, float *__restrict__ grad,
                                                    const double *__restrict__ lpartial, double *__restrict__ loss,
                                                    const double *__restrict__ spartial, double *__restrict__ stats) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < npar) {
        float acc = 0.f;
        for (int b = 0; b < nblocks; ++b) acc += gpartial[(size_t)b * npar + i];
        grad[i] = acc;
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x >= 252) {               // four idle-ish lanes of the last block: the scalars
        const int j = threadIdx.x - 252;                                    // 0: loss, 1..3: sum A, sum A^2, n
        if (j == 0) { double acc = 0.0; for (int b = 0; b < nblocks; ++b) acc += lpartial[b]; *loss = acc; }
        else if (stats) { double acc = 0.0; for (int b = 0; b < nblocks; ++b) acc += spartial[(size_t)b * 3 + (j - 1)]; stats[j - 1] = acc; }
    }
}
// the diagnostics of one ppo_grad launch with DIAG (after k_reduce_all, which it does not replace): fixed-order sums of the loss
// and diagnostic partials into the step's fp64 record row (layout: include/mhppo.h, mhppo_ppo_grad_diag); the actor pass also
// writes its k3 sum as fp32 to kl_slot (the slot behind the pair's packed gradients, all-reduced with them)
__global__ void k_reduce_diag(const double *__restrict__ lpartial, const double *__restrict__ dpartial, int nblocks, int head,
                              double *__restrict__ row, float *__restrict__ kl_slot) {
    const int j = threadIdx.x;              // 0: loss, 1 .. kDiagW: the diagnostic columns
    if (j > kDiagW) return;
    double acc = 0.0;
    if (j == 0) for (int b = 0; b < nblocks; ++b) acc += lpartial[b];
    else for (int b = 0; b < nblocks; ++b) acc += dpartial[(size_t)b * kDiagW + (j - 1)];
    if (head == 0) {
        if (j == 0) row[1] = acc; else row[4 + j] = acc;           // critic loss; sum (R-V), (R-V)^2, R, R^2 -> row[5 .. 8]
    } else {
        if (j == 0) row[0] = acc; else if (j <= 3) row[1 + j] = acc;   // actor loss; sum k3, clipped, H -> row[2 .. 4]
        if (j == 1 && kl_slot) *kl_slot = (float)acc;
    }
}
__global__ void k_reduce_scalars(const double *__restrict__ partial, int nblocks, int width, double *__restrict__ out) {
    const int j = threadIdx.x;
    if (j >= width) return;
    double acc = 0.0;
    for (int b = 0; b < nblocks; ++b) acc += partial[(size_t)b * width + j];
    out[j] = acc;
}

// ---- GAE(gamma, lambda) returns of the cross / wait buffers (an option; the reference's estimator is k_returns) ----------
// One thread per (car, env) column m, reverse scan over t with V(s_T) = 0 and R_T = 0 (the episode ends at step T-1):
//   R_t = r_t + gamma * ((1 - lambda) * V_old(s_{t+1}) + lambda * R_{t+1}),   ret_t = (float)R_t,   A_t = ret_t - V_old(s_t)
// so A_t = sum_k (gamma lambda)^k delta_{t+k}.  The recursion is fp64 without contraction (__dmul_rn / __dadd_rn): at lambda = 1
// it is r_t + gamma * R_{t+1}, the operations of k_returns, and ret equals that reward-to-go bit for bit.  A is formed in fp32
// as the actor kernel forms it (rtg - V).  Columns with route -1 (car absent) are written +0 and read nothing.  Each CTA writes
// fp64 partials (sum A, sum A^2, n) of route 0 then route 1; k_reduce_gae adds them in a fixed order (no atomics).
// Every access of a step is coalesced over m; the kGaeUnroll loads of a batch of steps are independent (memory parallelism).
constexpr int kGaeBlock = 256, kGaeGridMax = 4096, kGaeUnroll = 8;    // grid: min(columns / 256, 8 per SM, 4096 = workspace rows)
__global__ void __launch_bounds__(kGaeBlock) k_gae(const float *__restrict__ rew, const float *__restrict__ V,
                                                   const int8_t *__restrict__ route, int T, int64_t CN, double gamma, double lambda,
                                                   float *__restrict__ ret, double *__restrict__ partial /* [grid][6] */) {
    __shared__ double red[kGaeBlock / 32];
    double st[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const double oml = 1.0 - lambda;
    for (int64_t m = (int64_t)blockIdx.x * kGaeBlock + threadIdx.x; m < CN; m += (int64_t)gridDim.x * kGaeBlock) {
        const int r = route[m];
        const bool on = r >= 0;         // an absent column runs the same scan on zeros (no divergence in the warp): R = +0 throughout
        double R = 0.0, Vn = 0.0, sA = 0.0, sAA = 0.0;
        for (int t0 = T - 1; t0 >= 0; t0 -= kGaeUnroll) {
            float rw[kGaeUnroll], v[kGaeUnroll];
#pragma unroll
            for (int u = 0; u < kGaeUnroll; ++u) {
                const int64_t s = (int64_t)(t0 - u) * CN + m;
                rw[u] = (on && t0 - u >= 0) ? rew[s] : 0.f;
                v[u] = (on && t0 - u >= 0) ? V[s] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < kGaeUnroll; ++u) {
                if (t0 - u < 0) break;
                R = __dadd_rn((double)rw[u], __dmul_rn(gamma, __dadd_rn(__dmul_rn(oml, Vn), __dmul_rn(lambda, R))));
                const float Rf = (float)R;
                ret[(int64_t)(t0 - u) * CN + m] = Rf;
                const double A = (double)(Rf - v[u]);
                sA += A; sAA += A * A;
                Vn = (double)v[u];
            }
        }
        if (r == 0) { st[0] += sA; st[1] += sAA; st[2] += (double)T; }
        else if (r == 1) { st[3] += sA; st[4] += sAA; st[5] += (double)T; }
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const double v = team_sum(st[j], red, threadIdx.x, kGaeBlock, 0);
        if (threadIdx.x == 0) partial[(size_t)blockIdx.x * 6 + j] = v;
    }
}
// fixed-order sum of the k_gae partials [n][6]: warp j adds column j (lane l takes rows l, l + 32, ..., then a shuffle tree),
// so the up to kGaeGridMax rows cost a few independent loads per lane instead of one serial chain
__global__ void __launch_bounds__(192) k_reduce_gae(const double *__restrict__ partial, int n, double *__restrict__ out) {
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc = 0.0;
    for (int b = lane; b < n; b += 32) acc += partial[(size_t)b * 6 + j];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if (lane == 0) out[j] = acc;
}

// ---- minibatch plan (an option, Algo_PPO(n_minibatches=B); the reference's update is full-batch) --------------------------
// In epoch e, column m = car*N + n (global env id g = env_id0 + n) goes to bucket
//   b(car, g, e) = (w0 * B) >> 32,   w0 = word 0 of Philox4x32-10(counter = (e*C + car, 3 | iteration << 8, g_lo, g_hi), key = seed)
// (stream 3 of the policy-noise contract, policy_block), so the buckets of an R-rank run are those of one rank holding all envs.
// Per epoch the plan is a stable counting sort of the columns by bucket, for three selections at once (s = 0 cross: route 0,
// 1 wait: route 1, 2 existing: exist != 0), plus the per-bucket counts of existing columns whose choice action is 0 / 1.
// Within a bucket the columns are in ascending m.  Integer arithmetic in a fixed order throughout: the shared-memory histogram's
// atomics add integers (order-free), and every list position comes from a scan or a warp ballot, never from an atomic.
//   k_mb_count   grid (tiles, E): per-tile histogram [5][B] of one epoch -> hist[e][s][tile][b]
//   k_mb_scan    grid (E, 5)    : per-bucket totals -> counts; exclusive scan over (b, tile) -> hist = each tile's base, offsets
//   k_mb_scatter grid (tiles, E): rounds of 256 columns in m order, warp w after warp w-1, lanes ranked by __match_any_sync
// Layouts: lists int32 [E][3][M], offsets int64 [E][3][B+1] (bucket b of selection s is lists[e][s][off[b] .. off[b+1])),
// counts int64 [E][5][B] (rows: cross, wait, existing, existing with action 0, with action 1), workspace int32 [E][5][64][B].
constexpr int kMbBlock = 256, kMbMaxTiles = 64, kMbMaxBuckets = 1024, kMbRows = 5;
struct MbPlanArgs {
    RolloutDims d;                       // N, C, env_id0 and the Philox key of the rollout
    const int8_t *route, *exist;
    const float *act_d;
    uint32_t iteration;
    int E, B, tiles;
    int64_t M, tile;                     // columns, columns per tile (a multiple of kMbBlock)
    int32_t *hist, *lists;
    int64_t *offsets, *counts;
};
__device__ __forceinline__ int mb_bucket(const MbPlanArgs &a, int e, int64_t m, int &car) {
    car = (int)(m / a.d.N);
    const int64_t n = m - (int64_t)car * a.d.N;
    const PhiloxBlock b = policy_block(a.d, n, (uint32_t)(e * a.d.C + car), 3u | (a.iteration << 8));
    return (int)(((uint64_t)b.w0 * (uint64_t)a.B) >> 32);
}
// selection flags of column m: bit s set if the column belongs to selection s (0 cross, 1 wait, 2 existing, 3 / 4 action 0 / 1)
__device__ __forceinline__ unsigned mb_flags(const MbPlanArgs &a, int64_t m) {
    const int r = a.route[m];
    const bool ex = a.exist[m] != 0;
    const float ad = a.act_d[m];
    return (r == 0 ? 1u : 0u) | (r == 1 ? 2u : 0u) | (ex ? 4u : 0u) | ((ex && ad == 0.f) ? 8u : 0u) | ((ex && ad == 1.f) ? 16u : 0u);
}
__global__ void __launch_bounds__(kMbBlock) k_mb_count(MbPlanArgs a) {
    __shared__ int h[kMbRows * kMbMaxBuckets];
    const int e = blockIdx.y, tile = blockIdx.x, B = a.B;
    for (int i = threadIdx.x; i < kMbRows * B; i += kMbBlock) h[i] = 0;
    __syncthreads();
    const int64_t m0 = (int64_t)tile * a.tile, m1 = (m0 + a.tile < a.M) ? m0 + a.tile : a.M;
    for (int64_t m = m0 + threadIdx.x; m < m1; m += kMbBlock) {
        const unsigned f = mb_flags(a, m);
        if (!f) continue;
        int car;
        const int b = mb_bucket(a, e, m, car);
#pragma unroll
        for (int s = 0; s < kMbRows; ++s)
            if (f & (1u << s)) atomicAdd(&h[s * B + b], 1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kMbRows * B; i += kMbBlock) {
        const int s = i / B, b = i - s * B;
        a.hist[(((size_t)e * kMbRows + s) * kMbMaxTiles + tile) * B + b] = h[i];
    }
}
__global__ void __launch_bounds__(kMbMaxBuckets) k_mb_scan(MbPlanArgs a) {
    __shared__ int64_t wsum[kMbMaxBuckets / 32];
    const int e = blockIdx.x, s = blockIdx.y, B = a.B, b = threadIdx.x, lane = b & 31, w = b >> 5;
    int32_t *h = a.hist + ((size_t)e * kMbRows + s) * kMbMaxTiles * B;
    int64_t tot = 0;
    if (b < B)
        for (int t = 0; t < a.tiles; ++t) tot += h[(size_t)t * B + b];
    if (b < B) a.counts[((size_t)e * kMbRows + s) * B + b] = tot;
    if (s >= 3) return;                  // action counts: totals only
    // exclusive scan of tot over b (warp shuffles, then the warp sums)
    int64_t inc = tot;
    for (int o = 1; o < 32; o <<= 1) { const int64_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
        int64_t x = wsum[lane], xi = x;
        for (int o = 1; o < 32; o <<= 1) { const int64_t v = __shfl_up_sync(0xffffffffu, xi, o); if (lane >= o) xi += v; }
        wsum[lane] = xi - x;             // exclusive prefix of the warp sums
    }
    __syncthreads();
    if (b >= B) return;
    int64_t base = wsum[w] + inc - tot;
    int64_t *off = a.offsets + ((size_t)e * 3 + s) * (B + 1);
    off[b] = base;
    if (b == B - 1) off[B] = base + tot;
    for (int t = 0; t < a.tiles; ++t) { const int v = h[(size_t)t * B + b]; h[(size_t)t * B + b] = (int32_t)base; base += v; }
}
__global__ void __launch_bounds__(kMbBlock) k_mb_scatter(MbPlanArgs a) {
    __shared__ int run[3 * kMbMaxBuckets];
    const int e = blockIdx.y, tile = blockIdx.x, B = a.B, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 3 * B; i += kMbBlock) {
        const int s = i / B, b = i - s * B;
        run[i] = a.hist[(((size_t)e * kMbRows + s) * kMbMaxTiles + tile) * B + b];
    }
    __syncthreads();
    const int64_t m0 = (int64_t)tile * a.tile, m1 = (m0 + a.tile < a.M) ? m0 + a.tile : a.M;
    const unsigned lt = (1u << lane) - 1u;
    for (int64_t r0 = m0; r0 < m1; r0 += kMbBlock) {          // the same trip count in every thread of the CTA
        const int64_t m = r0 + threadIdx.x;
        const unsigned f = (m < m1) ? mb_flags(a, m) : 0u;
        int car, b = 0;
        if (f & 7u) b = mb_bucket(a, e, m, car);
        int key[3], pos[3] = {0, 0, 0};
        unsigned peers[3];
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            key[s] = (f & (1u << s)) ? b : -1;
            peers[s] = __match_any_sync(0xffffffffu, key[s]);
        }
        for (int w = 0; w < kMbBlock / 32; ++w) {             // warps in m order: warp w takes its slots after warp w - 1
            if (warp == w) {
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int leader = __ffs(peers[s]) - 1;
                    int base = 0;
                    if (lane == leader && key[s] >= 0) { base = run[s * B + key[s]]; run[s * B + key[s]] = base + __popc(peers[s]); }
                    pos[s] = __shfl_sync(0xffffffffu, base, leader) + __popc(peers[s] & lt);
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int s = 0; s < 3; ++s)
            if (key[s] >= 0) a.lists[((size_t)e * 3 + s) * a.M + pos[s]] = (int32_t)m;
    }
}

// ---- 6. Adam (torch.optim.Adam defaults, PY:719-724): p -= step_size * m / (sqrt(v) * inv_sqrt_bc2 + eps) ----
__global__ void __launch_bounds__(256) k_adam(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                                              float *__restrict__ v, int n, float beta1, float beta2, float step_size,
                                              float inv_sqrt_bc2, float eps, float grad_scale) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i] * grad_scale;
    const float mi = beta1 * m[i] + (1.0f - beta1) * gi;                 // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;            // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi; v[i] = vi;
    p[i] = p[i] - step_size * (mi / (sqrtf(vi) * inv_sqrt_bc2 + eps));
}

// both Adam steps of one epoch (actor and critic of a pair act on different nets, PY:810-815) in one launch
struct AdamArgs { float *p; const float *g; float *m, *v; int n; float step_size, inv_sqrt_bc2; };
__global__ void __launch_bounds__(256) k_adam2(AdamArgs a0, AdamArgs a1, float beta1, float beta2, float eps) {
    const AdamArgs a = blockIdx.y ? a1 : a0;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= a.n) return;
    const float gi = a.g[i];
    const float mi = beta1 * a.m[i] + (1.0f - beta1) * gi;
    const float vi = beta2 * a.v[i] + (1.0f - beta2) * gi * gi;
    a.m[i] = mi; a.v[i] = vi;
    a.p[i] = a.p[i] - a.step_size * (mi / (sqrtf(vi) * a.inv_sqrt_bc2 + eps));
}

// both Adam steps of a pair with the target-KL halt (Algo_PPO(target_kl=delta)): *kl_sum = the pair's actor k3 sum over all
// ranks (the fp32 slot behind its packed gradients); once it exceeds kl_limit = 1.5 delta n the pair is halted (*halt = 1) and
// this and every later launch of the update leave p, m, v untouched.  Every block takes the same decision: a block that reads the
// flag still 0 reads the same slot, and only a block that finds the limit exceeded writes the flag.  A step taken sets *taken = 1.
// The element arithmetic is k_adam2's.
__global__ void __launch_bounds__(256) k_adam2_halt(AdamArgs a0, AdamArgs a1, float beta1, float beta2, float eps,
                                                    const float *__restrict__ kl_sum, double kl_limit, int *halt, double *taken) {
    if (*(volatile int *)halt) return;
    if ((double)*kl_sum > kl_limit) { if (threadIdx.x == 0) *(volatile int *)halt = 1; return; }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *taken = 1.0;
    const AdamArgs a = blockIdx.y ? a1 : a0;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= a.n) return;
    const float gi = a.g[i];
    const float mi = beta1 * a.m[i] + (1.0f - beta1) * gi;
    const float vi = beta2 * a.v[i] + (1.0f - beta2) * gi * gi;
    a.m[i] = mi; a.v[i] = vi;
    a.p[i] = a.p[i] - a.step_size * (mi / (sqrtf(vi) * a.inv_sqrt_bc2 + eps));
}

// both Adam steps of a pair with per-network gradient-norm clipping (Algo_PPO(max_grad_norm=g)), torch's clip_grad_norm_ on each
// net: norm = ||g||_2 over the net's whole flat gradient, coef = max_norm / (norm + 1e-6), and the step uses coef * g when coef < 1.
// A non-finite norm (or max_norm = inf) gives coef = 1, the unclipped step.  One CTA per net (blockIdx.y), since the norm must be
// known before any element steps: pass 1 sums g^2 in fp64 (each thread a fixed strided subset, then a shuffle tree per warp and
// warp 0 over the warp sums: a fixed order, repeatable bit for bit), pass 2 is k_adam2's element arithmetic on g * coef (exact
// for coef = 1, so an unclipped step is k_adam2's bit for bit).  g is not written.  norms_out[y] = norm when norms_out != NULL.
// HALT: k_adam2_halt's halt on top, tested after the norms are written, so a step the halt skips still reports its norm.
// ADAPT: the KL-adaptive learning rate (Algo_PPO(lr_schedule="adaptive")), see AdaptArgs; a.step_size is then ignored.
constexpr int kClipBlock = 1024;

// rsl_rl's adaptive rule on each net's fp32 lr state lr[y], decided by thread 0 of net y's CTA after the halt test: kl = *kl_sum / n
// (the pair's all-reduced actor k3 sum over the step's n samples);
// kl > 2 delta: lr = max(1e-5, lr / 1.5); else 0 < kl < delta / 2: lr = min(1e-2, lr * 1.5); otherwise (NaN, +-inf included) the
// lr stays.  Each change is computed in fp64 and rounded to fp32; the step then uses step_size = (float)((double)lr / bc1[y]), the
// host's formula, so a step whose lr did not change is k_adam2's bit for bit.  lrs_out[y] (may be NULL) = the lr the step used.
struct AdaptArgs { float *lr; const float *kl_sum; double *lrs_out; double n, desired_kl, bc1[2]; };

template <bool HALT, bool ADAPT = false>
__global__ void __launch_bounds__(kClipBlock) k_adam2_clip(AdamArgs a0, AdamArgs a1, float beta1, float beta2, float eps, double max_norm,
                                                           double *__restrict__ norms_out, const float *__restrict__ kl_sum,
                                                           double kl_limit, int *halt, double *taken, AdaptArgs ad = AdaptArgs{}) {
    __shared__ double wsum[kClipBlock / 32];
    __shared__ float coef_s, step_s;
    const AdamArgs a = blockIdx.y ? a1 : a0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double ss = 0.0;
    for (int i = threadIdx.x; i < a.n; i += kClipBlock) { const double gi = (double)a.g[i]; ss += gi * gi; }
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_down_sync(0xffffffffu, ss, o);
    if (lane == 0) wsum[warp] = ss;
    __syncthreads();
    if (warp == 0) {
        double t = wsum[lane];
        for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
        if (lane == 0) {
            const double norm = sqrt(t), c = max_norm / (norm + 1e-6);
            coef_s = (isfinite(norm) && c < 1.0) ? (float)c : 1.0f;
            if (norms_out) norms_out[blockIdx.y] = norm;
        }
    }
    __syncthreads();
    if (HALT) {
        if (*(volatile int *)halt) return;
        if ((double)*kl_sum > kl_limit) { if (threadIdx.x == 0) *(volatile int *)halt = 1; return; }
        if (blockIdx.y == 0 && threadIdx.x == 0) *taken = 1.0;
    }
    if (ADAPT) {
        if (threadIdx.x == 0) {
            const double kl = (double)*ad.kl_sum / ad.n;
            float lr = ad.lr[blockIdx.y];
            if (isfinite(kl)) {
                if (kl > 2.0 * ad.desired_kl) lr = (float)fmax(1e-5, (double)lr / 1.5);
                else if (kl > 0.0 && kl < 0.5 * ad.desired_kl) lr = (float)fmin(1e-2, (double)lr * 1.5);
            }
            ad.lr[blockIdx.y] = lr;
            if (ad.lrs_out) ad.lrs_out[blockIdx.y] = (double)lr;
            step_s = (float)((double)lr / (blockIdx.y ? ad.bc1[1] : ad.bc1[0]));
        }
        __syncthreads();
    }
    const float coef = coef_s, step_size = ADAPT ? step_s : a.step_size;
    for (int i = threadIdx.x; i < a.n; i += kClipBlock) {
        const float gi = a.g[i] * coef;
        const float mi = beta1 * a.m[i] + (1.0f - beta1) * gi;
        const float vi = beta2 * a.v[i] + (1.0f - beta2) * gi * gi;
        a.m[i] = mi; a.v[i] = vi;
        a.p[i] = a.p[i] - step_size * (mi / (sqrtf(vi) * a.inv_sqrt_bc2 + eps));
    }
}

}  // namespace mhppo
