// QMIX monotonic mixer (network/mixer.py:21-80), forward + backward, optionally fused with the
// target mixer and the TD loss (algorithm/q_learner.py:161-168).
//
//   hy = s . wcat^T + bcat        one GEMM for the four hyper-network heads (linear_fwd), C = N*E+3E
//   one warp per (b,t) sample, lane = embed index e (E = 32):
//     hid_e = elu(sum_n q_n |w1[n,e]| + b1_e);  q_tot = sum_e hid_e |w2_e| + (sum_e relu(hb2_e) wb2_e + bb2)
//   the agents x embed contraction lives in registers, the embed reduction is a warp shuffle;
//   backward in the same warp emits the per-sample gradient row dhy[C] that feeds the
//   weight-gradient GEMM dwcat += dhy^T . s.
// Other embed widths E (qmix_hidden_dim, 1..128, marl_qmix_params.embed) run qmix_mix_kernel_e<J>: the lane owns the
// embed slots lane + 32 j, j < J = ceil(E / 32).
#include "linear.h"
#include "forkjoin.h"
#include "../../include/marl_b200.h"
#include "profile.h"
#include "tgemm.h"

#ifdef MARL_MIX_TRACE
// (select.cuh's optional stamps write into the kernel's trace through these file-scope device variables: one warp traces)
__device__ long long* g_mix_trace_ptr = nullptr;
#define MIX_SEL_STAMP(tag)                                                                                      \
    do {                                                                                                        \
        if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 300) && g_mix_trace_ptr) {                     \
            long long* t__ = g_mix_trace_ptr + (blockIdx.x ? 512 : 0);                                           \
            long long now__; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now__));                           \
            const int n__ = (int)t__[510]; if (n__ < 60) { t__[2 * n__] = (tag); t__[2 * n__ + 1] = now__; t__[510] = n__ + 1; } \
        }                                                                                                       \
    } while (0)
#endif
#include "select.cuh"

namespace marl {

constexpr int E = MARL_QMIX_EMBED;
#ifndef MARL_QMIX_WARPS
#define MARL_QMIX_WARPS 8
#endif
constexpr int kQmixWarps = MARL_QMIX_WARPS;        // samples (warps) per CTA
constexpr int kQmixCtasPerSm = 32 / kQmixWarps;    // 32 resident warps per SM at 64 registers
constexpr int kQmixMaxAgents = 64;
constexpr int kQmixMaxEmbed = MARL_QMIX_MAX_EMBED;   // qmix_hidden_dim: up to 4 embed slots per lane of qmix_mix_kernel_e

// Resident CTAs per SM of the instantiation with J embed slots per lane: a lane keeps ~7 floats per slot live across
// the sample (pre-activation, hidden, |w2|, relu(b2.0) inputs, both hyper_b2.2 weights, its gradient), so the wider
// instantiations get 80 (J = 2) and 128 (J = 3, 4) registers instead of 64.
__host__ __device__ constexpr int qmix_ctas_per_sm(int J) { return J == 1 ? kQmixCtasPerSm : (J == 2 ? 3 : 2); }

enum { QMIX_FWD = 0, QMIX_BWD = 1, QMIX_TD = 2 };

struct QmixMixArgs {
    int M, N, A, mode;
    const float* hy;  const float* q;  const float* wb2;  const float* bb2;            // eval side
    const float* hy_t; const float* q_t; const float* wb2_t; const float* bb2_t;       // target side (TD)
    const float* r; const float* term; const float* padded; float gamma;
    const float* dq_tot_in;       // BWD
    float* q_tot; float* q_tot_t;
    float* dhy;                   // [M,C]
    float* dq_small;              // [M,N] or null
    const long long* u; float* dq_dense;   // [M,N,A] or null
    const float* fc2_w; float* dhext;      // agent head W2 [A,H] and dL/dh through it [M,N,H], or null
    SelectArgs sel;                        // fused action-value selection (TD mode): q / q_t are then OUTPUTS
    float* g_wb2; float* g_bb2; float* scalars;
    long long* trace;                      // debug (marl_tgemm_trace, -DMARL_MIX_TRACE builds): globaltimer stamps of one warp
};
#ifdef MARL_MIX_TRACE
#define MIX_STAMP(tag) MIX_SEL_STAMP(tag)
#else
#define MIX_STAMP(tag) do { } while (0)
#endif

// forward of one sample for one lane; returns q_tot (all lanes) and the lane's intermediates
__device__ __forceinline__ float qmix_forward_lane(const float* __restrict__ y, const float* __restrict__ q, int N,
                                                   float wb2e, float bb2, int lane, float& pre, float& hid,
                                                   float& w2raw, float& hb2) {
    float acc = y[N * E + lane];                                   // hyper_b1
#pragma unroll 4
    for (int n = 0; n < N; ++n) acc = fmaf(q[n], fabsf(y[n * E + lane]), acc);   // bmm(q, |w1|) + b1, mixer.py:64-70
    pre = acc;
    hid = acc > 0.0f ? acc : (expf(acc) - 1.0f);                   // F.elu
    w2raw = y[N * E + E + lane];
    hb2 = y[N * E + 2 * E + lane];
    float part = hid * fabsf(w2raw) + fmaxf(hb2, 0.0f) * wb2e;     // bmm(hidden, |w2|) + hyper_b2(s), mixer.py:72-78
    return warp_sum(part) + bb2;
}

// (qmix_mix_kernel_e<J> below is the same kernel for the other embed widths: a change to one belongs in both)
__global__ void __launch_bounds__(kQmixWarps * 32, kQmixCtasPerSm) qmix_mix_kernel(QmixMixArgs a) {
#ifdef MARL_MIX_TRACE
    if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 300)) g_mix_trace_ptr = a.trace;      // (same value from both writers)
#endif
    MIX_STAMP(0);
    pdl_enter();
    MIX_STAMP(1);
    __shared__ float sdq[kQmixWarps][kQmixMaxAgents];
    __shared__ float sred[kQmixWarps][E + 1];
    __shared__ float ssel[kQmixWarps][2][kQmixMaxAgents];
    extern __shared__ __align__(16) float ssel_dyn[];         // fused selection: select_warp_floats() per warp
    const float* heads = nullptr;
    if (a.sel.q && a.sel.heads) {
        // this warp's first sample: its hidden rows are on their way (cp.async) while the CTA stages the head matrices
        const int m_first = blockIdx.x * kQmixWarps + (threadIdx.x >> 5);
        if (m_first < a.M)
            warp_stage_hidden_async(a.sel, m_first, a.N, a.A, threadIdx.x & 31, ssel_dyn + (threadIdx.x >> 5) * select_warp_floats(a.N, a.A, true));
        float* h = ssel_dyn + kQmixWarps * select_warp_floats(a.N, a.A, true);
        stage_heads(a.sel, a.A, h);
        heads = h;
        __syncthreads();
    }
    bool prestaged = a.sel.q && a.sel.heads;
    MIX_STAMP(2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = a.N, C = N * E + 3 * E;
    const float wb2e = a.wb2[lane], bb2 = a.bb2[0];
    float wb2te = 0.f, bb2t = 0.f;
    if (a.mode == QMIX_TD) { wb2te = a.wb2_t[lane]; bb2t = a.bb2_t[0]; }
    float acc_wb2 = 0.f, acc_bb2 = 0.f, acc_sq = 0.f, acc_mask = 0.f;
    for (int m = blockIdx.x * kQmixWarps + warp; m < a.M; m += gridDim.x * kQmixWarps) {
        const float* __restrict__ y = a.hy + (long long)m * C;
        const float* q = a.q + (long long)m * N;
        const float* qt = a.q_t + (long long)m * N;
        if (a.sel.q) {
            warp_select(a.sel, m, N, a.A, lane, ssel_dyn + warp * select_warp_floats(N, a.A, a.sel.heads), ssel[warp][0], ssel[warp][1], heads, prestaged);
            prestaged = false;
            q = ssel[warp][0]; qt = ssel[warp][1];
        }
        MIX_STAMP(3);
        float pre, hid, w2raw, hb2;
        const float tot = qmix_forward_lane(y, q, N, wb2e, bb2, lane, pre, hid, w2raw, hb2);
        if (lane == 0 && a.q_tot) a.q_tot[m] = tot;
        MIX_STAMP(4);
        if (a.mode == QMIX_FWD) continue;
        float G;
        if (a.mode == QMIX_TD) {
            float p2, h2, w2t, hbt;
            const float tot_t = qmix_forward_lane(a.hy_t + (long long)m * C, qt, N, wb2te, bb2t,
                                                  lane, p2, h2, w2t, hbt);
            if (lane == 0 && a.q_tot_t) a.q_tot_t[m] = tot_t;
            const float mask = 1.0f - a.padded[m];                                   // q_learner.py:83
            const float yt = a.r[m] + a.gamma * tot_t * (1.0f - a.term[m]);          // :165
            const float d = mask * (yt - tot);                                       // :166-167
            acc_sq += d * d; acc_mask += mask;                                       // (lane-uniform)
            G = -2.0f * mask * d;
        } else {
            G = a.dq_tot_in[m];
        }
        MIX_STAMP(5);
        // backward
        float* __restrict__ dy = a.dhy + (long long)m * C;
        const float dpre = G * fabsf(w2raw) * (pre > 0.0f ? 1.0f : (hid + 1.0f));   // elu'(x) = exp(x) for x <= 0
        const float sgn2 = (w2raw > 0.0f) ? 1.0f : (w2raw < 0.0f ? -1.0f : 0.0f);
        dy[N * E + lane] = dpre;                                                    // d hyper_b1
        dy[N * E + E + lane] = G * hid * sgn2;                                      // d hyper_w2 (through abs)
        dy[N * E + 2 * E + lane] = (hb2 > 0.0f) ? G * wb2e : 0.0f;                  // d hyper_b2.0 (through relu)
        acc_wb2 += G * fmaxf(hb2, 0.0f);
        acc_bb2 += G;
#pragma unroll 4
        for (int n = 0; n < N; ++n) {
            const float w1raw = y[n * E + lane];
            const float sgn1 = (w1raw > 0.0f) ? 1.0f : (w1raw < 0.0f ? -1.0f : 0.0f);
            dy[n * E + lane] = dpre * q[n] * sgn1;                                  // d hyper_w1 (through abs)
            const float dqn = warp_sum(dpre * fabsf(w1raw));
            if (lane == 0) sdq[warp][n] = dqn;
        }
        __syncwarp();
        MIX_STAMP(6);
        if (a.dq_small)
            for (int n = lane; n < N; n += 32) a.dq_small[(long long)m * N + n] = sdq[warp][n];
        if (a.dq_dense) {
            const int A = a.A;
            for (int i = lane; i < N * A; i += 32) {
                const int n = i / A, c = i - n * A;
                a.dq_dense[(long long)m * N * A + i] = (c == (int)a.u[(long long)m * N + n]) ? sdq[warp][n] : 0.0f;
            }
        }
        if (a.dhext) warp_dhext(a.fc2_w, a.u, m, N, lane, sdq[warp], a.dhext);
        __syncwarp();
        MIX_STAMP(7);
    }
    if (a.mode == QMIX_FWD) return;
    // block reduction of the hyper_b2.2 gradient and the loss scalars
    sred[warp][lane] = acc_wb2;
    if (lane == 0) sred[warp][E] = acc_bb2;
    __syncthreads();
    if (warp == 0) {
        float v = 0.f, b = 0.f;
        for (int w = 0; w < kQmixWarps; ++w) { v += sred[w][lane]; b += sred[w][E]; }
        if (a.g_wb2) atomicAdd(a.g_wb2 + lane, v);
        if (lane == 0 && a.g_bb2) atomicAdd(a.g_bb2, b);
    }
    if (a.mode == QMIX_TD) {
        __syncthreads();
        if (lane == 0) { sred[warp][0] = acc_sq; sred[warp][1] = acc_mask; }
        __syncthreads();
        if (threadIdx.x == 0) {
            float v = 0.f, b = 0.f;
            for (int w = 0; w < kQmixWarps; ++w) { v += sred[w][0]; b += sred[w][1]; }
            atomicAdd(a.scalars, v); atomicAdd(a.scalars + 1, b);
        }
    }
    MIX_STAMP(8);
}

// qmix_forward_lane for any E: the lane owns the embed slots e = lane + 32 j, j < J = ceil(E / 32); the slots at or past E
// are masked (they hold zeros and write nothing)
template <int J>
__device__ __forceinline__ float qmix_forward_slots(const float* __restrict__ y, const float* __restrict__ q, int N, int E,
                                                   const float (&wb2e)[J], float bb2, int lane, float (&pre)[J],
                                                   float (&hid)[J], float (&w2raw)[J], float (&hb2)[J]) {
    float acc[J];
#pragma unroll
    for (int j = 0; j < J; ++j) acc[j] = (lane + 32 * j < E) ? y[N * E + lane + 32 * j] : 0.0f;       // hyper_b1
#pragma unroll 4
    for (int n = 0; n < N; ++n)
#pragma unroll
        for (int j = 0; j < J; ++j)
            if (lane + 32 * j < E) acc[j] = fmaf(q[n], fabsf(y[n * E + lane + 32 * j]), acc[j]);   // bmm(q, |w1|) + b1, mixer.py:64-70
    float part;
#pragma unroll
    for (int j = 0; j < J; ++j) {
        const bool ok = (lane + 32 * j < E);
        const int e = lane + 32 * j;
        pre[j] = acc[j];
        hid[j] = acc[j] > 0.0f ? acc[j] : (expf(acc[j]) - 1.0f);              // F.elu
        w2raw[j] = ok ? y[N * E + E + e] : 0.0f;
        hb2[j] = ok ? y[N * E + 2 * E + e] : 0.0f;
        const float pj = hid[j] * fabsf(w2raw[j]) + fmaxf(hb2[j], 0.0f) * wb2e[j];   // bmm(hidden, |w2|) + hyper_b2(s), mixer.py:72-78
        part = j ? part + pj : pj;
    }
    return warp_sum(part) + bb2;
}

// qmix_mix_kernel for any other embed width E (1..128, E != 32): the same per-sample warp, J = ceil(E / 32) slots per lane.
// (E = 32 keeps qmix_mix_kernel above: routed through this template its instruction schedule changes.  The two are the same
// algorithm -- a change to one belongs in both; tests/test_qmix_embed_gpu.py runs E = 31 / 33 against E = 32 on inputs where
// they must agree.)
template <int J>
__global__ void __launch_bounds__(kQmixWarps * 32, qmix_ctas_per_sm(J)) qmix_mix_kernel_e(QmixMixArgs a, int E) {
    static_assert(J >= 1 && J * 32 <= kQmixMaxEmbed, "embed slots per lane");
#ifdef MARL_MIX_TRACE
    if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 300)) g_mix_trace_ptr = a.trace;      // (same value from both writers)
#endif
    MIX_STAMP(0);
    pdl_enter();
    MIX_STAMP(1);
    __shared__ float sdq[kQmixWarps][kQmixMaxAgents];
    __shared__ float sred[kQmixWarps][32 * J + 1];           // hyper_b2.2 weight gradient per slot | its bias at 32 J
    __shared__ float ssel[kQmixWarps][2][kQmixMaxAgents];
    extern __shared__ __align__(16) float ssel_dyn[];         // fused selection: select_warp_floats() per warp
    const float* heads = nullptr;
    if (a.sel.q && a.sel.heads) {
        // this warp's first sample: its hidden rows are on their way (cp.async) while the CTA stages the head matrices
        const int m_first = blockIdx.x * kQmixWarps + (threadIdx.x >> 5);
        if (m_first < a.M)
            warp_stage_hidden_async(a.sel, m_first, a.N, a.A, threadIdx.x & 31, ssel_dyn + (threadIdx.x >> 5) * select_warp_floats(a.N, a.A, true));
        float* h = ssel_dyn + kQmixWarps * select_warp_floats(a.N, a.A, true);
        stage_heads(a.sel, a.A, h);
        heads = h;
        __syncthreads();
    }
    bool prestaged = a.sel.q && a.sel.heads;
    MIX_STAMP(2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = a.N, C = N * E + 3 * E;
    float wb2e[J], wb2te[J], acc_wb2[J];
#pragma unroll
    for (int j = 0; j < J; ++j) wb2e[j] = (lane + 32 * j < E) ? a.wb2[lane + 32 * j] : 0.f;
    const float bb2 = a.bb2[0];
#pragma unroll
    for (int j = 0; j < J; ++j) wb2te[j] = 0.f;
    float bb2t = 0.f;
    if (a.mode == QMIX_TD) {
#pragma unroll
        for (int j = 0; j < J; ++j) wb2te[j] = (lane + 32 * j < E) ? a.wb2_t[lane + 32 * j] : 0.f;
        bb2t = a.bb2_t[0];
    }
#pragma unroll
    for (int j = 0; j < J; ++j) acc_wb2[j] = 0.f;
    float acc_bb2 = 0.f, acc_sq = 0.f, acc_mask = 0.f;
    for (int m = blockIdx.x * kQmixWarps + warp; m < a.M; m += gridDim.x * kQmixWarps) {
        const float* __restrict__ y = a.hy + (long long)m * C;
        const float* q = a.q + (long long)m * N;
        const float* qt = a.q_t + (long long)m * N;
        if (a.sel.q) {
            warp_select(a.sel, m, N, a.A, lane, ssel_dyn + warp * select_warp_floats(N, a.A, a.sel.heads), ssel[warp][0], ssel[warp][1], heads, prestaged);
            prestaged = false;
            q = ssel[warp][0]; qt = ssel[warp][1];
        }
        MIX_STAMP(3);
        float pre[J], hid[J], w2raw[J], hb2[J];
        const float tot = qmix_forward_slots<J>(y, q, N, E, wb2e, bb2, lane, pre, hid, w2raw, hb2);
        if (lane == 0 && a.q_tot) a.q_tot[m] = tot;
        MIX_STAMP(4);
        if (a.mode == QMIX_FWD) continue;
        float G;
        if (a.mode == QMIX_TD) {
            float p2[J], h2[J], w2t[J], hbt[J];
            const float tot_t = qmix_forward_slots<J>(a.hy_t + (long long)m * C, qt, N, E, wb2te, bb2t,
                                                         lane, p2, h2, w2t, hbt);
            if (lane == 0 && a.q_tot_t) a.q_tot_t[m] = tot_t;
            const float mask = 1.0f - a.padded[m];                                   // q_learner.py:83
            const float yt = a.r[m] + a.gamma * tot_t * (1.0f - a.term[m]);          // :165
            const float d = mask * (yt - tot);                                       // :166-167
            acc_sq += d * d; acc_mask += mask;                                       // (lane-uniform)
            G = -2.0f * mask * d;
        } else {
            G = a.dq_tot_in[m];
        }
        MIX_STAMP(5);
        // backward
        float* __restrict__ dy = a.dhy + (long long)m * C;
        float dpre[J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            dpre[j] = 0.f;
            if (lane + 32 * j >= E) continue;
            const int e = lane + 32 * j;
            dpre[j] = G * fabsf(w2raw[j]) * (pre[j] > 0.0f ? 1.0f : (hid[j] + 1.0f));   // elu'(x) = exp(x) for x <= 0
            const float sgn2 = (w2raw[j] > 0.0f) ? 1.0f : (w2raw[j] < 0.0f ? -1.0f : 0.0f);
            dy[N * E + e] = dpre[j];                                                   // d hyper_b1
            dy[N * E + E + e] = G * hid[j] * sgn2;                                     // d hyper_w2 (through abs)
            dy[N * E + 2 * E + e] = (hb2[j] > 0.0f) ? G * wb2e[j] : 0.0f;              // d hyper_b2.0 (through relu)
            acc_wb2[j] += G * fmaxf(hb2[j], 0.0f);
        }
        acc_bb2 += G;
#pragma unroll 4
        for (int n = 0; n < N; ++n) {
            float t;
#pragma unroll
            for (int j = 0; j < J; ++j) {
                float v = 0.f;
                if (lane + 32 * j < E) {
                    const int e = lane + 32 * j;
                    const float w1raw = y[n * E + e];
                    const float sgn1 = (w1raw > 0.0f) ? 1.0f : (w1raw < 0.0f ? -1.0f : 0.0f);
                    dy[n * E + e] = dpre[j] * q[n] * sgn1;                             // d hyper_w1 (through abs)
                    v = dpre[j] * fabsf(w1raw);
                }
                t = j ? t + v : v;
            }
            const float dqn = warp_sum(t);
            if (lane == 0) sdq[warp][n] = dqn;
        }
        __syncwarp();
        MIX_STAMP(6);
        if (a.dq_small)
            for (int n = lane; n < N; n += 32) a.dq_small[(long long)m * N + n] = sdq[warp][n];
        if (a.dq_dense) {
            const int A = a.A;
            for (int i = lane; i < N * A; i += 32) {
                const int n = i / A, c = i - n * A;
                a.dq_dense[(long long)m * N * A + i] = (c == (int)a.u[(long long)m * N + n]) ? sdq[warp][n] : 0.0f;
            }
        }
        if (a.dhext) warp_dhext(a.fc2_w, a.u, m, N, lane, sdq[warp], a.dhext);
        __syncwarp();
        MIX_STAMP(7);
    }
    if (a.mode == QMIX_FWD) return;
    // block reduction of the hyper_b2.2 gradient and the loss scalars
#pragma unroll
    for (int j = 0; j < J; ++j) sred[warp][lane + 32 * j] = acc_wb2[j];
    if (lane == 0) sred[warp][32 * J] = acc_bb2;
    __syncthreads();
    if (warp == 0) {
        float v[J], b = 0.f;
#pragma unroll
        for (int j = 0; j < J; ++j) v[j] = 0.f;
        for (int w = 0; w < kQmixWarps; ++w) {
#pragma unroll
            for (int j = 0; j < J; ++j) v[j] += sred[w][lane + 32 * j];
            b += sred[w][32 * J];
        }
#pragma unroll
        for (int j = 0; j < J; ++j)
            if (a.g_wb2 && lane + 32 * j < E) atomicAdd(a.g_wb2 + lane + 32 * j, v[j]);
        if (lane == 0 && a.g_bb2) atomicAdd(a.g_bb2, b);
    }
    if (a.mode == QMIX_TD) {
        __syncthreads();
        if (lane == 0) { sred[warp][0] = acc_sq; sred[warp][1] = acc_mask; }
        __syncthreads();
        if (threadIdx.x == 0) {
            float v = 0.f, b = 0.f;
            for (int w = 0; w < kQmixWarps; ++w) { v += sred[w][0]; b += sred[w][1]; }
            atomicAdd(a.scalars, v); atomicAdd(a.scalars + 1, b);
        }
    }
    MIX_STAMP(8);
}

// The hy GEMMs write / read rows of pitch C = N E + 3 E.  When C * 4 bytes is not a multiple of 16 the rows are not
// TMA-addressable: such an hy stays on the register-staged kernels of linear.cu even with the TMA back end switched on
// (whose builders would otherwise still take the other operands and store hy through their scalar epilogue).
static bool hy_tma(int N, int E) { return ((N * E + 3 * E) & 3) == 0; }

static int hyper_fwd(int M, int N, int S, int E, const marl_qmix_params* p, const float* s, float* hy, cudaStream_t st) {
    LinearFwd f{};
    f.in = plain_operand(s, S, S);
    f.w = p->wcat; f.ldw = S; f.bias = p->bcat;
    f.y = hy; f.ldy = N * E + 3 * E; f.M = M; f.N = N * E + 3 * E; f.batch = 1;
    return linear_fwd(f, st, hy_tma(N, E));
}

static int hyper_wgrad(int M, int N, int S, int E, const float* s, const float* dhy, const marl_qmix_grads* g, cudaStream_t st) {
    LinearWgrad w{};
    w.dy = dhy; w.lddy = N * E + 3 * E; w.in = plain_operand(s, S, S);
    w.dw = g->wcat; w.ldw = S; w.db = g->bcat; w.M = M; w.N = N * E + 3 * E; w.batch = 1;
    return linear_wgrad(w, st, hy_tma(N, E));
}

// two_hyper_layers = True (network/mixer.py:36-43): hyper_w1 = Linear(S, hh) - ReLU - Linear(hh, N*E), hyper_w2 likewise
// with E outputs; hyper_b1 / hyper_b2 keep one layer.  h [M, 2 hh] holds the two hidden layers (after the ReLU) for
// the backward; the outputs land in the same hy layout [w1 | b1 | w2 | b2.0] the mixing kernel reads.
static int hyper2_fwd(int M, int N, int S, int E, const marl_qmix_hyper2* p, const float* s, float* h, float* hy, cudaStream_t st) {
    const int hh = p->hh, C = N * E + 3 * E;
    const bool tma = hy_tma(N, E);
    int rc;
    LinearFwd f{};
    f.in = plain_operand(s, S, S); f.w = p->w_in; f.ldw = S; f.bias = p->b_in;
    f.y = h; f.ldy = 2 * hh; f.M = M; f.N = 2 * hh; f.relu = 1; f.batch = 1;
    if ((rc = linear_fwd(f, st))) return rc;
    LinearFwd a{};
    a.in = plain_operand(h, 2 * hh, hh); a.w = p->w1_out; a.ldw = hh; a.bias = p->b1_out;
    a.y = hy; a.ldy = C; a.M = M; a.N = N * E; a.batch = 1;
    if ((rc = linear_fwd(a, st, tma))) return rc;
    LinearFwd b{};
    b.in = plain_operand(h + hh, 2 * hh, hh); b.w = p->w2_out; b.ldw = hh; b.bias = p->b2_out;
    b.y = hy + N * E + E; b.ldy = C; b.M = M; b.N = E; b.batch = 1;
    if ((rc = linear_fwd(b, st, tma))) return rc;
    LinearFwd c{};
    c.in = plain_operand(s, S, S); c.w = p->w_b1; c.ldw = S; c.bias = p->b_b1;
    c.y = hy + N * E; c.ldy = C; c.M = M; c.N = E; c.batch = 1;
    if ((rc = linear_fwd(c, st, tma))) return rc;
    LinearFwd e{};
    e.in = plain_operand(s, S, S); e.w = p->w_b20; e.ldw = S; e.bias = p->b_b20;
    e.y = hy + N * E + 2 * E; e.ldy = C; e.M = M; e.N = E; e.batch = 1;
    return linear_fwd(e, st, tma);
}

// gradients of everything in front of hy, given dhy [M, C]; dh [M, 2 hh] workspace
static int hyper2_bwd(int M, int N, int S, int E, const marl_qmix_hyper2* p, const float* s, const float* h, const float* dhy,
                      float* dh, const marl_qmix_hyper2_grads* g, cudaStream_t st) {
    const int hh = p->hh, C = N * E + 3 * E;
    const bool tma = hy_tma(N, E);
    int rc;
    LinearWgrad w{};                     // hyper_b1
    w.dy = dhy + N * E; w.lddy = C; w.in = plain_operand(s, S, S); w.dw = g->w_b1; w.ldw = S; w.db = g->b_b1; w.M = M; w.N = E; w.batch = 1;
    if ((rc = linear_wgrad(w, st, tma))) return rc;
    w.dy = dhy + N * E + 2 * E; w.dw = g->w_b20; w.db = g->b_b20;     // hyper_b2.0
    if ((rc = linear_wgrad(w, st, tma))) return rc;
    LinearWgrad o1{};                    // hyper_w1.2
    o1.dy = dhy; o1.lddy = C; o1.in = plain_operand(h, 2 * hh, hh); o1.dw = g->w1_out; o1.ldw = hh; o1.db = g->b1_out; o1.M = M; o1.N = N * E; o1.batch = 1;
    if ((rc = linear_wgrad(o1, st, tma))) return rc;
    LinearWgrad o2{};                    // hyper_w2.2
    o2.dy = dhy + N * E + E; o2.lddy = C; o2.in = plain_operand(h + hh, 2 * hh, hh); o2.dw = g->w2_out; o2.ldw = hh; o2.db = g->b2_out; o2.M = M; o2.N = E; o2.batch = 1;
    if ((rc = linear_wgrad(o2, st, tma))) return rc;
    LinearDgrad d1{};                    // dh[:, :hh] = (dhy_w1 . W1.2) * (h > 0)
    d1.dy = dhy; d1.lddy = C; d1.w = p->w1_out; d1.ldw = hh; d1.dx = dh; d1.lddx = 2 * hh; d1.relu_src = h; d1.ldrs = 2 * hh;
    d1.M = M; d1.N = N * E; d1.K = hh; d1.batch = 1;
    if ((rc = linear_dgrad(d1, st, tma))) return rc;
    LinearDgrad d2{};                    // dh[:, hh:] = (dhy_w2 . W2.2) * (h > 0)
    d2.dy = dhy + N * E + E; d2.lddy = C; d2.w = p->w2_out; d2.ldw = hh; d2.dx = dh + hh; d2.lddx = 2 * hh; d2.relu_src = h + hh; d2.ldrs = 2 * hh;
    d2.M = M; d2.N = E; d2.K = hh; d2.batch = 1;
    if ((rc = linear_dgrad(d2, st, tma))) return rc;
    LinearWgrad i{};                     // the two first layers as one [2 hh, S] problem
    i.dy = dh; i.lddy = 2 * hh; i.in = plain_operand(s, S, S); i.dw = g->w_in; i.ldw = S; i.db = g->b_in; i.M = M; i.N = 2 * hh; i.batch = 1;
    return linear_wgrad(i, st);
}

// grid-stride launch: at most one wave of the instantiation's resident CTAs
static int mix_grid(int M, int ctas_per_sm) {
    int blocks = (M + kQmixWarps - 1) / kQmixWarps;
    return blocks < 1 ? 1 : (blocks > ctas_per_sm * kNumSMs ? ctas_per_sm * kNumSMs : blocks);
}

template <auto kern, class... Args>
static void launch_mix_kernel(int ctas_per_sm, size_t dyn, cudaStream_t st, const QmixMixArgs& a, Args... extra) {
    // A launch whose static + dynamic shared memory passes 48 KB needs the opt-in.  The static part is the kernel's own (it grows
    // with the slots per lane: sred), so it is read from the kernel; unknown, the opt-in is made for any dynamic size.
    static size_t static_smem = 0;
    static bool known = false, attr_set = false;        // (one set per kernel)
    if (!known) {
        cudaFuncAttributes fa{};
        if (cudaFuncGetAttributes(&fa, kern) == cudaSuccess) static_smem = fa.sharedSizeBytes;
        else { cudaGetLastError(); static_smem = 48 * 1024; }
        known = true;
    }
    if (dyn > 0 && dyn + static_smem > 48 * 1024 && !attr_set) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSelectSmemMax);
        attr_set = true;
    }
    launch_pdl(kern, dim3(mix_grid(a.M, ctas_per_sm)), dim3(kQmixWarps * 32), dyn, st, a, extra...);
}

// the mixing kernel for embed width E (1..128): E = 32 has its own kernel, the others ceil(E / 32) slots per lane
static int launch_mix(const QmixMixArgs& a, int E, size_t dyn, cudaStream_t st) {
    ProfScope ps_("qmix_mix_kernel", st);
    switch (E == 32 ? 0 : (E + 31) / 32) {
        case 0: launch_mix_kernel<qmix_mix_kernel>(kQmixCtasPerSm, dyn, st, a); break;
        case 1: launch_mix_kernel<qmix_mix_kernel_e<1>>(qmix_ctas_per_sm(1), dyn, st, a, E); break;
        case 2: launch_mix_kernel<qmix_mix_kernel_e<2>>(qmix_ctas_per_sm(2), dyn, st, a, E); break;
        case 3: launch_mix_kernel<qmix_mix_kernel_e<3>>(qmix_ctas_per_sm(3), dyn, st, a, E); break;
        case 4: launch_mix_kernel<qmix_mix_kernel_e<4>>(qmix_ctas_per_sm(4), dyn, st, a, E); break;
        default: return MARL_EINVAL;
    }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

}  // namespace marl

using namespace marl;

static bool qmix_params_ok(const marl_qmix_params* p) { return p && p->wcat && p->bcat && p->wb2 && p->bb2; }

// qmix_hidden_dim of a struct: 0 means 32 (zero-initialised callers from before the field existed); -1 when out of range
static int embed_of(int embed) {
    const int E = embed == 0 ? 32 : embed;
    return (E >= 1 && E <= kQmixMaxEmbed) ? E : -1;
}

extern "C" int marl_qmix_fwd(int M, int N, int S, const marl_qmix_params* p, const float* q, const float* s, float* hy,
                             float* q_tot, void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !qmix_params_ok(p) || !q || !s || !hy || !q_tot) return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = hyper_fwd(M, N, S, E, p, s, hy, st);
    if (rc) return rc;
    QmixMixArgs a{};
    a.M = M; a.N = N; a.mode = QMIX_FWD; a.hy = hy; a.q = q; a.wb2 = p->wb2; a.bb2 = p->bb2; a.q_tot = q_tot;
    return launch_mix(a, E, 0, st);
}

extern "C" int marl_qmix_bwd(int M, int N, int S, const marl_qmix_params* p, const float* q, const float* s,
                             const float* hy, const float* dq_tot, float* dhy, float* dq, const marl_qmix_grads* g,
                             void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !qmix_params_ok(p) || !q || !s || !hy || !dq_tot || !dhy || !g)
        return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0 || embed_of(g->embed) != E) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    QmixMixArgs a{};
    a.M = M; a.N = N; a.mode = QMIX_BWD; a.hy = hy; a.q = q; a.wb2 = p->wb2; a.bb2 = p->bb2;
    a.dq_tot_in = dq_tot; a.dhy = dhy; a.dq_small = dq; a.g_wb2 = g->wb2; a.g_bb2 = g->bb2;
    int rc = launch_mix(a, E, 0, st);
    if (rc) return rc;
    return hyper_wgrad(M, N, S, E, s, dhy, g, st);
}

extern "C" int marl_qmix_td_fwd_bwd(const marl_dims* d, const marl_qmix_params* p, const marl_qmix_params* pt,
                                    const float* s, const float* s_next, float* q_chosen, float* q_tc,
                                    const long long* u, const float* r, const float* terminated, const float* padded,
                                    float gamma, float* hy, float* hy_target, float* dhy, float* q_tot, float* q_tot_target,
                                    float* dq, const marl_qmix_grads* g, float* scalars, int flags, const float* fc2_w,
                                    float* dhext, const marl_select_fused* sel, void* stream) {
    if (!d || !p || !pt || !p->wb2 || !p->bb2 || !pt->wb2 || !pt->bb2 || !s || !s_next || !q_chosen || !q_tc || !r ||
        !terminated || !padded || !hy || !hy_target || !dhy || !g || !scalars)
        return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0 || embed_of(pt->embed) != E || embed_of(g->embed) != E) return MARL_EINVAL;
    if (!(flags & 1) && (!p->wcat || !p->bcat || !pt->wcat || !pt->bcat)) return MARL_EINVAL;   // hyper GEMMs run here
    if (!(flags & 2) && (!g->wcat || !g->bcat)) return MARL_EINVAL;
    if ((dq || dhext || sel) && !u) return MARL_EINVAL;
    if (sel && !select_ok(sel)) return MARL_EINVAL;
    if (dhext && (!fc2_w || ((uintptr_t)fc2_w & 7) || ((uintptr_t)dhext & 7))) return MARL_EINVAL;
    if (d->N < 1 || d->N > kQmixMaxAgents || d->S < 1) return MARL_EINVAL;
    const int M = d->B * d->L;
    if (M <= 0) return MARL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    pdl_scope((long long)M * d->N);
    int rc;
    if (!(flags & 1)) {
        ForkJoin fj(st, 2);      // eval and target hyper-networks side by side
        if ((rc = hyper_fwd(M, d->N, d->S, E, p, s, hy, fj.lane(0)))) return rc;
        if ((rc = hyper_fwd(M, d->N, d->S, E, pt, s_next, hy_target, fj.lane(1)))) return rc;
        fj.join();
    }
    QmixMixArgs a{};
    a.M = M; a.N = d->N; a.A = d->A; a.mode = QMIX_TD;
    a.hy = hy; a.q = q_chosen; a.wb2 = p->wb2; a.bb2 = p->bb2;
    a.hy_t = hy_target; a.q_t = q_tc; a.wb2_t = pt->wb2; a.bb2_t = pt->bb2;
    a.r = r; a.term = terminated; a.padded = padded; a.gamma = gamma;
    a.q_tot = q_tot; a.q_tot_t = q_tot_target; a.dhy = dhy; a.u = u; a.dq_dense = dq;
    a.fc2_w = fc2_w; a.dhext = dhext;
    if (sel) a.sel = select_args(sel, u, q_chosen, q_tc);
    a.g_wb2 = g->wb2; a.g_bb2 = g->bb2; a.scalars = scalars;
    a.trace = trace_buffer();
    const size_t dyn = sel ? select_smem(kQmixWarps, d->N, d->A, sel->hidden_evals != nullptr) : 0;
    if (dyn > kSelectSmemMax) return MARL_EINVAL;
    if ((rc = launch_mix(a, E, dyn, st))) return rc;
    if (flags & 2) return MARL_OK;
    return hyper_wgrad(M, d->N, d->S, E, s, dhy, g, st);
}

extern "C" int marl_qmix_mix_fwd(int M, int N, const marl_qmix_params* p, const float* q, const float* hy, float* q_tot,
                                 void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || !p || !p->wb2 || !p->bb2 || !q || !hy || !q_tot) return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    QmixMixArgs a{};
    a.M = M; a.N = N; a.mode = QMIX_FWD; a.hy = hy; a.q = q; a.wb2 = p->wb2; a.bb2 = p->bb2; a.q_tot = q_tot;
    return launch_mix(a, E, 0, (cudaStream_t)stream);
}

extern "C" int marl_qmix_mix_bwd(int M, int N, const marl_qmix_params* p, const float* q, const float* hy,
                                 const float* dq_tot, float* dhy, float* dq, const marl_qmix_grads* g, void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || !p || !p->wb2 || !p->bb2 || !q || !hy || !dq_tot || !dhy || !g) return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0 || embed_of(g->embed) != E) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    QmixMixArgs a{};
    a.M = M; a.N = N; a.mode = QMIX_BWD; a.hy = hy; a.q = q; a.wb2 = p->wb2; a.bb2 = p->bb2;
    a.dq_tot_in = dq_tot; a.dhy = dhy; a.dq_small = dq; a.g_wb2 = g->wb2; a.g_bb2 = g->bb2;
    return launch_mix(a, E, 0, (cudaStream_t)stream);
}

static bool hyper2_ok(const marl_qmix_hyper2* p) {
    return p && p->hh > 0 && p->w_in && p->b_in && p->w1_out && p->b1_out && p->w2_out && p->b2_out && p->w_b1 && p->b_b1 &&
           p->w_b20 && p->b_b20;
}

extern "C" int marl_qmix_hyper2_fwd(int M, int N, int S, const marl_qmix_hyper2* p, const float* s, float* h, float* hy,
                                    void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !hyper2_ok(p) || !s || !h || !hy) return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    return hyper2_fwd(M, N, S, E, p, s, h, hy, (cudaStream_t)stream);
}

extern "C" int marl_qmix_hyper2_bwd(int M, int N, int S, const marl_qmix_hyper2* p, const float* s, const float* h,
                                    const float* dhy, float* dh, const marl_qmix_hyper2_grads* g, void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !hyper2_ok(p) || !s || !h || !dhy || !dh || !g || !g->w_in ||
        !g->b_in || !g->w1_out || !g->b1_out || !g->w2_out || !g->b2_out || !g->w_b1 || !g->b_b1 || !g->w_b20 || !g->b_b20)
        return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    return hyper2_bwd(M, N, S, E, p, s, h, dhy, dh, g, (cudaStream_t)stream);
}

extern "C" int marl_qmix_hyper_fwd(int M, int N, int S, const marl_qmix_params* p, const float* s, float* hy, void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !qmix_params_ok(p) || !s || !hy) return MARL_EINVAL;
    const int E = embed_of(p->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    pdl_scope((long long)M * N);
    return hyper_fwd(M, N, S, E, p, s, hy, (cudaStream_t)stream);
}

extern "C" int marl_qmix_hyper_wgrad(int M, int N, int S, const float* s, const float* dhy, const marl_qmix_grads* g,
                                     void* stream) {
    if (M < 0 || N < 1 || N > kQmixMaxAgents || S < 1 || !s || !dhy || !g || !g->wcat || !g->bcat) return MARL_EINVAL;
    const int E = embed_of(g->embed);
    if (E < 0) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    pdl_scope((long long)M * N);
    return hyper_wgrad(M, N, S, E, s, dhy, g, (cudaStream_t)stream);
}

/* Can the fused mixing kernels (csrc/qmix.cu, csrc/select_td.cu) stage the selection (heads = 0) / the selection plus the
 * agents' heads (heads = 1) of an [N, A] problem in shared memory?  1 / 0; the host gates its launch plan on this instead
 * of repeating the kernels' build-time constants. */
extern "C" int marl_select_fits(int qmix, int N, int A, int heads) {
    if (N <= 0 || A <= 0) return 0;
    return marl::select_smem(qmix ? marl::kQmixWarps : 8, N, A, heads != 0) <= marl::kSelectSmemMax ? 1 : 0;
}
