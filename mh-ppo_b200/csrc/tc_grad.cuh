// tc_grad.cuh -- the fused forward + loss + backward kernel of the PPO update with the forward pass and
// backward-data on the 5th-generation tensor cores (13-input nets: cross / wait actors and critics).
//
// Same contract as k_ppo_grad<16, HEAD> (ppo_update.cuh), which stays as the exact-fp32 cross-check and serves the wider
// choice nets.  One persistent 256-thread CTA per SM walks 128-sample tiles; in warps 0-3 thread = sample = TMEM lane.
//   forward       D[128 x J] = A[128 x K] * W[J x K]^T         (tc_mlp.cuh: 3xTF32, hi/lo operand tiles, fp32 in TMEM)
//   (layers 1-3; the 32 -> 4 output layer and its backward-data are 2 x 128 FFMAs per sample on the CUDA cores)
//   backward-data dIn[128 x K] = delta[128 x J] * W[J x K]     = the same MMA shapes with B = the FLAT transposed weights
//                 Wt[k][j] read as an [N = K rows][reduction = J] K-major tile (BwdTiles)
//   weight grad   dWt[k][j] += sum_s in[s][k] * delta[s][j]    FFMA register tiles (WgradAcc) on fp32 rows in shared memory:
//                 the reduction runs over samples, which a tf32 MMA could only read from 128B-swizzled MN-major tiles
//                 (tc.cuh); it runs on four dedicated warps CONCURRENTLY with the chain of backward-data MMAs and their
//                 epilogues (ReLU masks kept in registers from the forward pass) on the other four.
// The next tile's features / loss inputs / column index are fetched with cp.async into the unused layer-4 tile space.
// Every epilogue writes its row twice: fp32 into the row buffer (weight gradient) and hi/lo into the next A operand tile.
#pragma once
#include "ppo_update.cuh"
#include "tc_kernels.cuh"

namespace mhppo {

// B operands of backward-data: tile element (row = k, reduction index = j) = W[j][k] = Wt[k][j] (flat layout, mlp.cuh)
struct BwdTiles {
    static constexpr int W4 = H3 * tcm::OUTP, W3 = H2 * H3, W2 = H1 * H2;      // [32 x 16], [64 x 32], [32 x 64]
    static constexpr int FLOATS = 2 * (W4 + W3 + W2);
    float *w4h, *w4l, *w3h, *w3l, *w2h, *w2l;
    __device__ void carve(float *p) { w4h = p; p += W4; w4l = p; p += W4; w3h = p; p += W3; w3l = p; p += W3; w2h = p; p += W2; w2l = p; }
    template <int KP>
    __device__ void stage(const float *__restrict__ g) {
        auto fill = [&](float *h, float *l, const float *wt, int N, int J, int Jsrc) {   // wt[k * Jsrc + j], k < N, j < Jsrc, zero-padded to J
            for (int i = threadIdx.x; i < N * J; i += blockDim.x) {
                const int k = i / J, j = i % J;
                const float v = (j < Jsrc) ? wt[k * Jsrc + j] : 0.f, hv = tcm::hi_part(v);
                h[tc::tile_index(k, j, J)] = hv; l[tc::tile_index(k, j, J)] = v - hv;
            }
        };
        fill(w4h, w4l, g + off_w4(KP), H3, tcm::OUTP, OP);
        fill(w3h, w3l, g + off_w3(KP), H2, H3, H3);
        fill(w2h, w2l, g + off_w2(KP), H1, H2, H2);
    }
};

// NC columns [col0, col0 + NC) of this thread's row of the A operand, split hi / lo, into tensor memory
template <int NC>
__device__ __forceinline__ void put_tmem(uint32_t a_hi, uint32_t a_lo, const float *v) {
    float t[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) t[j] = tcm::hi_part(v[j]);
    if (NC == 32) tc::tmem_st32(a_hi, reinterpret_cast<const float (&)[32]>(t)); else tc::tmem_st16(a_hi, reinterpret_cast<const float (&)[16]>(t));
#pragma unroll
    for (int j = 0; j < NC; ++j) t[j] = v[j] - tcm::hi_part(v[j]);
    if (NC == 32) tc::tmem_st32(a_lo, reinterpret_cast<const float (&)[32]>(t)); else tc::tmem_st16(a_lo, reinterpret_cast<const float (&)[16]>(t));
}
// one thread issues the 3xTF32 chains of a layer with the A operand in tensor memory (hi at a_hi, lo at a_lo: K columns each)
template <int K, int J>
__device__ __forceinline__ void issue_layer_ts(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, const float *bh, const float *bl, uint64_t *bar) {
    constexpr uint32_t idesc = tc::make_idesc_tf32(128, J);
    const uint32_t b0 = tc::smem_u32(bh), b1 = tc::smem_u32(bl);
    bool acc = false;
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t pa = (pass == 1) ? a_lo : a_hi, pb = (pass == 2) ? b1 : b0;
#pragma unroll
        for (int k0 = 0; k0 < K; k0 += 8) {
            tc::mma_tf32_ts(d_tmem, pa + k0, tc::make_desc(pb + (k0 / 4) * 128, K), idesc, acc);
            acc = true;
        }
    }
    tc::mma_commit(bar);
}

constexpr int kTcGradRow = 16 + H1 + H2 + H3 + OP;       // 148 floats: 16-byte aligned rows, stride = 20 (mod 32) words -> conflict-free 128-bit accesses
constexpr int kTcGradNetFloats = (tcm::NetTiles<16>::FLOATS + 255) & ~255;
constexpr int kTcGradStageExtra = 256;             // the part of the fetch staging area that does not fit the unused layer-4 tiles
constexpr size_t kTcGradSmemFloats = (size_t)kTcGradNetFloats + BwdTiles::FLOATS + (size_t)2 * 128 * kTcGradRow + kTcGradStageExtra;      // two row buffers

// Warp-specialised CTA: warps 0-3 ("E", thread = sample = TMEM lane) issue the MMAs and run the epilogues; warps 4-7 ("W")
// only accumulate the weight gradient.  The two groups hand the row buffer back and forth through named barriers:
//   R_l (E -> W): the rows now hold what the weight gradient of layer l needs;  F_l (W -> E): layer l has been read, its
//   input-activation columns may be overwritten by the delta of the layer below.
// E keeps a freshly computed delta in registers, feeds it to the tensor core through the A tile at once, and stores it into
// the rows only when W releases them, so the chain of backward-data MMAs runs ahead of the (longer) weight-gradient chain.
constexpr int kTcGradE = 128, kTcGradW = 128, kTcGradBlock = kTcGradE + kTcGradW;
enum { BAR_E = 1, BAR_W = 10, BAR_R4 = 2, BAR_F4 = 3, BAR_R3 = 4, BAR_F3 = 5, BAR_R2 = 6, BAR_F2 = 7, BAR_R1 = 8, BAR_F1 = 9, BAR_F1B = 11 };   // F1 of odd tiles: BAR_F1B
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// (producer side of the PTX producer / consumer barrier pattern: shared-memory stores before bar.arrive are visible to the
// threads that leave the matching bar.sync, no extra fence needed)
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

template <int HEAD, bool DIAG = false>
__global__ void __launch_bounds__(kTcGradBlock, 1) k_ppo_grad_tc(SampleSet ss, const float *__restrict__ net, LossArgs la,
                                                              float *__restrict__ gpartial, double *__restrict__ lpartial,
                                                              int *__restrict__ fail_flag) {
    resolve_adv_stats(la);
    constexpr int KP = 16, ROW = kTcGradRow, NG = kTcGradW / 64, NT = kTcGradBlock;
    typedef WgradAcc<KP, NG> WG;
    extern __shared__ __align__(1024) float smem[];
    __shared__ TcShared sh;
    __shared__ double red[kTcGradBlock / 32];
    __shared__ __align__(16) float w4c[H3 + 4];                   // column 0 of Wt4 and b4[0], fp32 (the output layer runs on the CUDA cores)
    tcm::NetTiles<KP> w;
    BwdTiles bw;
    w.carve(smem);
    bw.carve(smem + kTcGradNetFloats);
    float *rows0 = smem + kTcGradNetFloats + BwdTiles::FLOATS;     // tile t lives in row buffer t & 1
    constexpr int RBUF = 128 * kTcGradRow;
    w.stage(net);
    bw.stage<KP>(net);
    // Landing area of the asynchronous fetch of the NEXT tile (cp.async: no destination registers, nothing for later
    // instructions to wait on), [array][thread]: the layer-4 operand tiles of both tile sets are never read by this kernel (the
    // output layer runs on the CUDA cores), 2 x 1024 floats, plus 256 floats of its own.
    float *stA = w.w4h;                                             // features 0..7
    float *stB = bw.w4h;                                            // features 8..12, rtg, V, old log-prob
    float *stC = rows0 + 2 * RBUF;                                  // action, compacted-column index of the tile after next
    static_assert(tcm::NetTiles<KP>::W4 == 512 && BwdTiles::W4 == 512, "staging area = the two unused layer-4 tile pairs");
    static_assert(HEAD == 0 || HEAD == 1, "single-output heads only: the categorical choice nets use k_ppo_grad");
    for (int i = threadIdx.x; i <= H3; i += blockDim.x) w4c[i] = (i < H3) ? net[off_w4(KP) + i * OP] : net[off_b4(KP)];
    // TMEM: forward accumulators in columns 0-63; each backward layer has its own columns, so a delta can be read a second time
    // (for the deferred row store) after the next MMA has been issued: layer 4 -> 64..95, layer 2 -> 96..127, layer 3 -> 128..191
    // A operands (activations / deltas, hi and lo halves) live in tensor memory too: columns 256..319 and 320..383
    constexpr uint32_t kCols = 512, C2 = 96, C3 = 128, AH = 256, AL = 320;
    if (threadIdx.x == 0) { tc::mbar_init(&sh.bar, 1); sh.fail = 0; }
    if ((threadIdx.x >> 5) == 0) tc::tmem_alloc(&sh.tmem_base, kCols);
    tc::fence_async_smem(); tc::fence_before(); __syncthreads(); tc::fence_after();
    const uint32_t tmem = sh.tmem_base;
    const int tid = threadIdx.x;
    const bool is_e = tid < kTcGradE;
    LossAcc acc;
    bool ok = true;
    const int64_t tile0 = (int64_t)blockIdx.x * 128, tstep = (int64_t)gridDim.x * 128;

    if (!is_e) {
        // ================= W: weight gradient of every layer, layer 4 first =================
        WG wg;
        wg.init(tid - kTcGradE);
        constexpr int PART = 128 / NG;                    // rows per group
        const int s0 = wg.half * PART;
        int t = 0;
        for (int64_t base = tile0; base < ss.Q; base += tstep, ++t) {
            const float *rows = rows0 + (t & 1) * RBUF;
            bar_sync(BAR_R4, NT);  wg.layer4(rows, ROW, s0, PART);             bar_arrive(BAR_F4, NT);
            bar_sync(BAR_R3, NT);  wg.layer3(rows, ROW, s0, PART);             bar_arrive(BAR_F3, NT);
            bar_sync(BAR_R2, NT);  wg.layer2(rows, ROW, s0, PART);             bar_arrive(BAR_F2, NT);
            bar_sync(BAR_R1, NT);  wg.layer1_and_biases(rows, ROW, s0, PART);  bar_arrive((t & 1) ? BAR_F1B : BAR_F1, NT);
        }
        float *rows = rows0;
        // add the groups in the (now dead) row buffer, fixed order: deterministic
        bar_sync(BAR_W, kTcGradW);
#pragma unroll 1
        for (int g = 0; g < NG; ++g) {
            if (wg.half == g) wg.emit(rows, g > 0);
            bar_sync(BAR_W, kTcGradW);
        }
    } else {
        // ================= E: MMA issue + epilogues =================
        const uint32_t trow = tmem + ((uint32_t)((tid >> 5) * 32) << 16);
        uint32_t phase = 0;
        auto sync_for_mma = [&]() { tc::tmem_wait_st(); tc::fence_before(); bar_sync(BAR_E, kTcGradE); tc::fence_after(); };
        const uint32_t ahi = trow + AH, alo = trow + AL;        // this warp's lanes of the A operand
        const uint32_t Ahi = tmem + AH, Alo = tmem + AL;        // operand addresses for the MMA (lane 0)
        auto wait_mma = [&]() { ok &= tc::mbar_wait(&sh.bar, phase); phase ^= 1; tc::fence_after(); };
        LossIn lin;
        lin.rtg = lin.V = lin.act = lin.logp = 0.f;
        // ---- asynchronous fetch.  issue(base, idx): the features and loss inputs of work item base + tid start their trip into
        // this thread's slots of the staging area; collect(): they are read back one tile later.  The compacted-column index a
        // tile needs for its addresses is itself fetched one tile earlier (slot stC[128 + tid]), so no address waits for a load.
        auto cp4 = [](float *dst, const void *src) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(tc::smem_u32(dst)), "l"(src) : "memory");
        };
        auto issue = [&](int64_t base, int32_t col, bool &sel, int64_t &s) {      // col: ss.idx[k] of this item (ignored without a list)
            const int64_t q = base + tid;
            sel = q < ss.Q;
            s = 0;
            if (sel) {
                const int64_t tt = q / ss.K, k = q - tt * ss.K;
                s = tt * ss.CN + (ss.idx ? (int64_t)col : k);
#pragma unroll
                for (int f = 0; f < 13; ++f)
                    if (f < ss.D) cp4((f < 8 ? stA + f * 128 : stB + (f - 8) * 128) + tid, ss.x + (int64_t)f * ss.S + s);
                cp4(stB + 5 * 128 + tid, la.rtg + s);
                if (HEAD != 0) { cp4(stB + 6 * 128 + tid, la.V + s); cp4(stB + 7 * 128 + tid, la.logp_old + s); }
                if (HEAD == 1) cp4(stC + tid, la.act + s);
            }
        };
        auto issue_col = [&](int64_t base) {                                       // the column index of work item base + tid
            const int64_t q = base + tid;
            if (ss.idx && q < ss.Q) cp4(stC + 128 + tid, ss.idx + (q % ss.K));
        };
        auto commit_wait = [&]() { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); };
        auto collect = [&](bool sel, float (&x)[KP]) {
#pragma unroll
            for (int f = 0; f < KP; ++f) x[f] = (sel && f < ss.D && f < 13) ? (f < 8 ? stA[f * 128 + tid] : stB[(f - 8) * 128 + tid]) : 0.f;
            if (sel) {
                lin.rtg = stB[5 * 128 + tid];
                if (HEAD != 0) { lin.V = stB[6 * 128 + tid]; lin.logp = stB[7 * 128 + tid]; }
                if (HEAD == 1) lin.act = stC[tid];
            }
        };
        float xn[KP];
        bool seln = false;
        int64_t sn = 0;
        {   // prologue: the first tile's column index with a plain load, then its data and the second tile's index in flight
            const int64_t q = tile0 + tid;
            const int32_t col0 = (ss.idx && q < ss.Q) ? ss.idx[q % ss.K] : 0;
            issue(tile0, col0, seln, sn);
            issue_col(tile0 + tstep);
        }
        int t = 0;
        for (int64_t base = tile0; base < ss.Q; base += tstep, ++t) {
            float *row = rows0 + (t & 1) * RBUF + (size_t)tid * ROW;
            // this tile's data (issued one tile ago) and the next tile's column index have landed; the next tile's data and the
            // index of the tile after it start their trip now and travel during the whole tile
            commit_wait();
            const bool sel = seln;
            const int64_t s = sn;
            collect(sel, xn);
            const LossIn lcur = lin;
            {
                const int32_t col1 = __float_as_int(stC[128 + tid]);
                issue(base + tstep, col1, seln, sn);
                issue_col(base + 2 * tstep);
            }
            float v[32];
            uint32_t m1 = 0, m2a = 0, m2b = 0, m3 = 0;                // ReLU masks of the three hidden layers
            // ---- forward.  This tile's row buffer still belongs to W (layer 1 + biases of the tile before the previous one) until its F1;
            // the previous tile's weight gradient runs on the other buffer meanwhile.
            put_tmem<KP>(ahi, alo, xn);
            sync_for_mma();
            if (tid == 0) issue_layer_ts<KP, H1>(tmem, Ahi, Alo, w.w1h, w.w1l, &sh.bar);
            if (t >= 2) bar_sync((t & 1) ? BAR_F1B : BAR_F1, NT);
#pragma unroll
            for (int k = 0; k < KP; k += 4) st4(row + WG::X + k, make_float4(xn[k], xn[k + 1], xn[k + 2], xn[k + 3]));
            wait_mma();
            tc::tmem_ld32(trow, v);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b = ld4(w.b1 + j);               // (the bias arrays are 16-byte aligned in the weight image)
                v[j] = fmaxf(v[j] + b.x, 0.f); v[j + 1] = fmaxf(v[j + 1] + b.y, 0.f); v[j + 2] = fmaxf(v[j + 2] + b.z, 0.f); v[j + 3] = fmaxf(v[j + 3] + b.w, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) m1 |= (v[j] > 0.f ? 1u : 0u) << j;
#pragma unroll
            for (int j = 0; j < 32; j += 4) st4(row + WG::A1 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
            put_tmem<32>(ahi, alo, v);
            sync_for_mma();
            if (tid == 0) issue_layer_ts<H1, H2>(tmem, Ahi, Alo, w.w2h, w.w2l, &sh.bar);
            wait_mma();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                tc::tmem_ld32(trow + 32 * h, v);
                uint32_t m = 0;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b = ld4(w.b2 + 32 * h + j);
                    v[j] = fmaxf(v[j] + b.x, 0.f); v[j + 1] = fmaxf(v[j + 1] + b.y, 0.f); v[j + 2] = fmaxf(v[j + 2] + b.z, 0.f); v[j + 3] = fmaxf(v[j + 3] + b.w, 0.f);
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) m |= (v[j] > 0.f ? 1u : 0u) << j;
                if (h) m2b = m; else m2a = m;
#pragma unroll
                for (int j = 0; j < 32; j += 4) st4(row + WG::A2 + 32 * h + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
                put_tmem<32>(ahi + 32 * h, alo + 32 * h, v);
            }
            sync_for_mma();
            if (tid == 0) issue_layer_ts<H2, H3>(tmem, Ahi, Alo, w.w3h, w.w3l, &sh.bar);
            wait_mma();
            tc::tmem_ld32(trow, v);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b = ld4(w.b3 + j);
                v[j] = fmaxf(v[j] + b.x, 0.f); v[j + 1] = fmaxf(v[j + 1] + b.y, 0.f); v[j + 2] = fmaxf(v[j + 2] + b.z, 0.f); v[j + 3] = fmaxf(v[j + 3] + b.w, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) m3 |= (v[j] > 0.f ? 1u : 0u) << j;
#pragma unroll
            for (int j = 0; j < 32; j += 4) st4(row + WG::A3 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
            // ---- output layer and its backward-data stay on the CUDA cores, exact fp32, from the registers that already hold a3,
            // instead of two more dependent MMA round trips per tile.  The 13-input nets (heads 0 and 1) have ONE output: only column
            // 0 of the padded 32 x 4 weight block is live, so this is 32 FFMAs forward and 32 FMULs backward per sample.
            {
                float o0 = w4c[H3];                                                                   // b4[0]
#pragma unroll
                for (int k4 = 0; k4 < H3 / 4; ++k4) {
                    const float4 wk = ld4(w4c + 4 * k4);                                              // Wt4[4 k4 .. 4 k4 + 3][0]
                    o0 = fmaf(v[4 * k4 + 0], wk.x, o0); o0 = fmaf(v[4 * k4 + 1], wk.y, o0);
                    o0 = fmaf(v[4 * k4 + 2], wk.z, o0); o0 = fmaf(v[4 * k4 + 3], wk.w, o0);
                }
                // ---- loss epilogue -> dz (an unselected row keeps dz = 0: every gradient term of it vanishes)
                float d4[OP] = {0.f, 0.f, 0.f, 0.f};
                if (sel) ppo_loss<HEAD, false, DIAG>(la, s, lcur, make_float4(o0, 0.f, 0.f, 0.f), d4, acc);
                st4(row + WG::D4, make_float4(d4[0], 0.f, 0.f, 0.f));
                bar_arrive(BAR_R4, NT);                       // a3 and dz are in the rows: dW4 on W
#pragma unroll
                for (int k4 = 0; k4 < H3 / 4; ++k4) {                                                 // delta3 = relu'(a3) * dz0 * W4[:, 0]
                    const float4 wk = ld4(w4c + 4 * k4);
                    v[4 * k4 + 0] = ((m3 >> (4 * k4 + 0)) & 1u) ? d4[0] * wk.x : 0.f; v[4 * k4 + 1] = ((m3 >> (4 * k4 + 1)) & 1u) ? d4[0] * wk.y : 0.f;
                    v[4 * k4 + 2] = ((m3 >> (4 * k4 + 2)) & 1u) ? d4[0] * wk.z : 0.f; v[4 * k4 + 3] = ((m3 >> (4 * k4 + 3)) & 1u) ? d4[0] * wk.w : 0.f;
                }
            }
            put_tmem<32>(ahi, alo, v);
            sync_for_mma();
            if (tid == 0) issue_layer_ts<H3, H2>(tmem + C3, Ahi, Alo, bw.w3h, bw.w3l, &sh.bar);
            bar_sync(BAR_F4, NT);                             // a3 has been read
#pragma unroll
            for (int j = 0; j < 32; j += 4) st4(row + WG::A3 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
            bar_arrive(BAR_R3, NT);                           // delta3 is in the rows
            // ---- layer 3: the 64 deltas go to the A tile now and are read from TMEM once more for the rows
            wait_mma();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                tc::tmem_ld32(trow + C3 + 32 * h, v);
                const uint32_t m = h ? m2b : m2a;
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = ((m >> j) & 1u) ? v[j] : 0.f;
                put_tmem<32>(ahi + 32 * h, alo + 32 * h, v);
            }
            sync_for_mma();
            if (tid == 0) issue_layer_ts<H2, H1>(tmem + C2, Ahi, Alo, bw.w2h, bw.w2l, &sh.bar);
            bar_sync(BAR_F3, NT);                             // a2 has been read
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                tc::tmem_ld32(trow + C3 + 32 * h, v);
                const uint32_t m = h ? m2b : m2a;
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    st4(row + WG::A2 + 32 * h + j, make_float4(((m >> j) & 1u) ? v[j] : 0.f, ((m >> (j + 1)) & 1u) ? v[j + 1] : 0.f,
                                                               ((m >> (j + 2)) & 1u) ? v[j + 2] : 0.f, ((m >> (j + 3)) & 1u) ? v[j + 3] : 0.f));
            }
            bar_arrive(BAR_R2, NT);                           // delta2 is in the rows
            // ---- layer 2
            wait_mma();
            tc::tmem_ld32(trow + C2, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = ((m1 >> j) & 1u) ? v[j] : 0.f;
            tc::fence_before();                               // TMEM reads are done before the next tile's MMAs (sync_for_mma follows)
            bar_sync(BAR_F2, NT);                             // a1 has been read
#pragma unroll
            for (int j = 0; j < 32; j += 4) st4(row + WG::A1 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
            bar_arrive(BAR_R1, NT);                           // delta1 is in the rows: layer 1 and the biases
        }
        asm volatile("cp.async.wait_all;" ::: "memory");     // (nothing is in flight past the last tile; belt and braces before the area is reused)
        // the last two tiles' rows have been read (one F1 arrival of W is still unmatched per buffer in use)
        if (t >= 2) bar_sync((t & 1) ? BAR_F1B : BAR_F1, NT);
        if (t >= 1) bar_sync(((t - 1) & 1) ? BAR_F1B : BAR_F1, NT);
    }
    // ================= emit the CTA's partials =================
    if (!ok) atomicExch(fail_flag, 1);
    __syncthreads();
    constexpr int NPAR = net_params(KP);
    float *gp = gpartial + (size_t)blockIdx.x * NPAR;
    for (int i = tid; i < NPAR; i += NT) gp[i] = rows0[i];
    const double lsum = team_sum(acc.loss, red, tid, NT, 0);
    if (tid == 0) lpartial[blockIdx.x] = lsum;
    if (HEAD == 0 && la.spartial) {
        const double t0 = team_sum(acc.sA, red, tid, NT, 0), t1 = team_sum(acc.sAA, red, tid, NT, 0), t2 = team_sum(acc.cnt, red, tid, NT, 0);
        if (tid == 0) { la.spartial[blockIdx.x * 3 + 0] = t0; la.spartial[blockIdx.x * 3 + 1] = t1; la.spartial[blockIdx.x * 3 + 2] = t2; }
    }
    if (DIAG) write_diag_partials(acc, la.dpartial, red, tid, NT);
    tc::fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) tc::tmem_dealloc(tmem, 512);
}

}  // namespace mhppo
