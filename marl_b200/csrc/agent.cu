// Shared-parameter recurrent agent (fc1 -> ReLU -> GRUCell -> fc2), unrolled over the episode.
// Replaces the per-timestep Python loop of controller/share_params.py:125-168 around
// network/q_network.py:16-21 and its autograd reversal.
//
//   phase A (all B*L*N rows at once):   x  = relu(fc1([obs | last_action | agent_id]))   (linear_fwd)
//                                       gi = W_ih x + b_ih                               (linear_fwd)
//   phase B (sequential in t):          persistent CTAs own R rows (b,n) each for all L steps;
//                                       a 64x4 thread grid keeps its slice of W_hh in registers,
//                                       h lives in shared memory, one __syncthreads per step.
//   phase C (all rows):                 q = W2 h + b2                                     (linear_fwd)
//
// Independent unrolls (eval on o, target on o_next) run in different CTAs of the same launch;
// dependent ones (the double-Q eval unroll on o_next that starts from the final hidden of the
// eval unroll on o, algorithm/q_learner.py:96,110) are chained inside the same CTA.
#include "linear.h"
#include "tgemm.h"
#include "front.h"
#include "forkjoin.h"
#include "../../include/marl_b200.h"
#include "profile.h"
#include <algorithm>
#include <memory>

namespace marl {

constexpr int kMaxStreams = 4;
constexpr int kGruPrio = -1;        // launch priority of the recurrence kernels (see launch_pdl_prio)
constexpr int kGruThreads = 128;   // 64 hidden units x 2-way split of the reduction, one warp per SM sub-partition
#ifndef MARL_GI_DEPTH
#define MARL_GI_DEPTH 4
#endif
#ifndef MARL_BWD_DEPTH
#define MARL_BWD_DEPTH 6
#endif
constexpr int kGiDepth = MARL_GI_DEPTH;   // cp.async ring depth (time steps) of the forward's input gates
constexpr int kGruGroups = 2;      // chains advanced side by side in one CTA (one 128-thread group each)
constexpr int kGruMaxRows = 8;     // rows per group and pass

// MUFU-based gate non-linearities: ex2.approx / rcp.approx are accurate to ~2 ulp, i.e. <= 2e-7 absolute on
// the (0,1) / (-1,1) outputs -- the same order as the fp32 rounding of the reference's own libm path.
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float gate_sigmoid(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float gate_tanh(float x) {
    // 1 - 2/(1 + e^2x) loses relative accuracy to cancellation near 0: switch to the odd Taylor polynomial there
    const float big = fmaf(-2.0f, rcp_approx(1.0f + ex2_approx(2.8853900817779268f * x)), 1.0f);
    const float x2 = x * x;
    const float small = x * fmaf(x2, fmaf(x2, fmaf(x2, -0.0539682540f, 0.1333333333f), -0.3333333333f), 1.0f);
    return fabsf(x) < 0.2f ? small : big;
}

// Packed FP32 pairs (sm_100 FFMA2): one instruction = two fused multiply-adds on an aligned register pair.  The recurrent
// loops run ONE warp per SM sub-partition, which issues an FFMA only every ~2.5 cycles (clock64 traces, profiles/README.md), so
// they are bound by instructions issued, not by FMA lanes: the (even k, odd k) partial sums the loops already kept apart become
// the two halves of one packed accumulator -- same products, same association, same rounding, half the instructions.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

struct GruSegment {
    const float* gi;      // [B,L,N,3H]
    const float* w_hh;    // [3H,H]
    const float* b_hh;    // [3H]
    float* hidden;        // [B,L,N,H]
    float* gates;         // [B,L,N,4H] or null
    float* h_last;        // [B*N,H] or null
    const int* ep_len;    // [B] or null: rows stop at their episode's length (padded steps are not computed)
};

struct GruFwdArgs {
    GruSegment seg[kMaxStreams];
    int chain_start[kMaxStreams];
    int chain_len[kMaxStreams];
    const float* h0[kMaxStreams];
    int n_chains, B, L, N;
    unsigned short rows_of[kMaxStreams][kNumSMs];   // rows of chain c advanced by CTA i (balanced on the host, see plan_rows)
    const int* row_order[kMaxStreams];              // per chain: logical position -> row (b*N + n), or null = identity (row_order_kernel)
    long long* trace;                                // debug (marl_tgemm_trace): clock64 phase stamps of steps 8..15, CTA 0 / CTA 100
    int agent_stride;                                // separated networks (SEP instantiation): floats from agent n's parameters to n+1's
};
#ifdef MARL_GRU_TRACE      // tools/gru_trace.py with an A/B build (tools/ab_build.py trace -DMARL_GRU_TRACE)
// (stamps of steps 8..15 stay in registers -- a store per stamp costs ~75 cycles and distorts the step -- and are written after the loop)
#define GRU_STAMP(tag)                                                                                                  \
    do {                                                                                                                \
        if (trace && t >= 8 && t < 16) stamp[(t - 8) * 6 + (tag)] = (unsigned)clock();                                  \
    } while (0)
#else
#define GRU_STAMP(tag) do { } while (0)
#endif

// One CTA advances R rows (b,n) of one chain through all its segments.  Thread (j, ks): hidden unit j,
// half ks of the 64-long reduction; its 3 x 32 W_hh weights stay in registers for the whole segment.
// 128-thread named barrier: the CTA hosts one such group per chain, each advancing its own rows
__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(kGruThreads) : "memory"); }

// Separated networks (one parameter set per agent, SEP): logical positions are dealt agent-major, position p = n*B + b is row
// b*N + n, and a pass never straddles two agents (gru_pass_rows), so the W_hh slice in registers is the pass's agent's.
template <bool SEP>
__device__ __forceinline__ int gru_position_row(int p, int B, int N) { return SEP ? (p % B) * N + p / B : p; }
template <bool SEP>
__device__ __forceinline__ int gru_pass_rows(int pos, int left, int B) {
    const int n = min(kGruMaxRows, left);
    return SEP ? min(n, B - pos % B) : n;
}

template <int R, bool SEP>
__device__ __forceinline__ void gru_chain_fwd(const GruFwdArgs& a, int chain, int row0, int nrows, float* smem, int bar_id) {
    float (*hs)[R][MARL_H] = reinterpret_cast<float (*)[R][MARL_H]>(smem);                          // [2][R][H]
    float (*ring)[R][MARL_G] = reinterpret_cast<float (*)[R][MARL_G]>(smem + 2 * R * MARL_H);       // [D][R][3H]
    const int tid = threadIdx.x & (kGruThreads - 1), ks = tid & 1, j = tid >> 1;
    const int L = a.L, N = a.N;
    // logical position (what the CTAs are dealt) -> row b*N + n: identity, or the length-sorted deal of row_order_kernel
    // (resolved once per pass into shared memory: the previous pass ended with a group barrier)
    __shared__ int srow_all[kGruGroups][kGruMaxRows];
    int* srow = srow_all[bar_id - 1];
    if (tid < R) {
        const int* order = a.row_order[chain];
        srow[tid] = (order && tid < nrows) ? __ldg(order + row0 + tid) : gru_position_row<SEP>(row0 + tid, a.B, N);
    }
    group_sync(bar_id);
    auto row_at = [&](int rr) { return srow[rr]; };
    constexpr int OWN = (R + 1) / 2;                  // rows whose gate math this lane owns: rr = ks + 2q
    bool own[OWN]; long long base[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int rr = ks + 2 * q, row = row_at(rr);
        own[q] = rr < nrows;
        base[q] = own[q] ? ((long long)(row / N) * L * N + (row % N)) : 0;
    }
    // cp.async work list: R rows x 48 chunks of 16 B per time step
    constexpr int NCH = (R * 48 + kGruThreads - 1) / kGruThreads;
    long long csrc[NCH]; int cdst[NCH];
#pragma unroll
    for (int l = 0; l < NCH; ++l) {
        const int c = tid + l * kGruThreads, rr = c / 48, ch = c % 48, row = row_at(rr);
        if (c < R * 48 && rr < nrows) {
            csrc[l] = ((long long)(row / N) * L * N + (row % N)) * MARL_G + ch * 4;
            cdst[l] = rr * MARL_G + ch * 4;
        } else { csrc[l] = -1; cdst[l] = 0; }
    }
#ifdef MARL_GRU_TRACE
    long long* trace = (a.trace && tid == 0 && chain == 0 && (blockIdx.x == 0 || blockIdx.x == 100)) ? a.trace + (blockIdx.x ? 512 : 0) : nullptr;
    unsigned stamp[48] = {};
    if (trace) { trace[508] = R; trace[509] = nrows; }
#endif
    const float* h0 = a.h0[chain];
    for (int idx = tid; idx < R * MARL_H; idx += kGruThreads) {
        const int rr = idx / MARL_H, jj = idx % MARL_H, row = row_at(rr);
        hs[0][rr][jj] = (h0 && rr < nrows) ? h0[(long long)row * MARL_H + jj] : 0.0f;
    }
    int cur = 0;
    for (int sg = a.chain_start[chain]; sg < a.chain_start[chain] + a.chain_len[chain]; ++sg) {
        const GruSegment S = a.seg[sg];
        const long long poff = SEP ? (long long)(row0 / a.B) * a.agent_stride : 0;      // this pass's agent
        const float* w_hh = S.w_hh + poff;
        const float* b_hh = S.b_hh + poff;
        f32x2 w[3][16];                                  // (w[k], w[k+1]) pairs of this lane's slice of rows g*H + j
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(w_hh + (long long)(g * MARL_H + j) * MARL_H + 4 * (2 * i + ks)));
                w[g][2 * i] = pack2(v.x, v.y); w[g][2 * i + 1] = pack2(v.z, v.w);
            }
        const float bh_r = __ldg(b_hh + j), bh_z = __ldg(b_hh + MARL_H + j), bh_n = __ldg(b_hh + 2 * MARL_H + j);
        // per-step output pointers of the rows this lane owns: advanced by one time step (N rows) per iteration
        float* hp[OWN]; float* gp_out[OWN];
#pragma unroll
        for (int q = 0; q < OWN; ++q) {
            hp[q] = S.hidden + base[q] * MARL_H + j;
            gp_out[q] = S.gates ? S.gates + base[q] * (4 * MARL_H) + j : nullptr;
        }
        const long long hstep = (long long)N * MARL_H, gstep = (long long)N * 4 * MARL_H;
        // (measured and dropped: the time loop of the one- and two-row passes unrolled by the ring depth, ring slots and h-buffer side as
        // compile-time constants -- the loop-back went from 90 to 28 cycles and the refill from 60 to 40 in the clock64 trace, the
        // two-row CTAs from 720 to ~635 cycles per step, but the CTAs that run a target group beside their eval row stayed at ~730
        // and the step got 2.5 us SLOWER (four times the code in two groups at different places: instruction cache))
        // early exit (SURVEY 8(f) N3): the rows of this pass advance in lock-step, so the pass runs to the longest of its episodes
        int Lp = L;
        if (S.ep_len) {
            Lp = 1;
            for (int rr = 0; rr < nrows; ++rr) Lp = max(Lp, min(L, __ldg(S.ep_len + row_at(rr) / N)));
        }
        auto issue = [&](int t) {
            if (t < Lp) {
#pragma unroll
                for (int l = 0; l < NCH; ++l)
                    if (csrc[l] >= 0) cp_async16(&ring[t % kGiDepth][0][0] + cdst[l], S.gi + csrc[l] + (long long)t * N * MARL_G);
            }
            cp_async_commit();
        };
#pragma unroll
        for (int t = 0; t < kGiDepth - 1; ++t) issue(t);
        for (int t = 0; t < Lp; ++t) {
            GRU_STAMP(0);
            cp_async_wait<kGiDepth - 2>();           // this thread's copies for step t have landed
            group_sync(bar_id);                      // ... the whole group's; also orders the h double buffer
            GRU_STAMP(1);
            // Few rows per CTA = latency-bound chain: the refill's address math and LSU hand-off (~150 cycles when it sat
            // here, measured with clock64) go behind the FMAs, where they overlap the FMA drain.  Many rows per CTA =
            // throughput-bound: keep the prefetch as early as possible.
            constexpr bool kLateIssue = R <= 2;
            if (!kLateIssue) issue(t + kGiDepth - 1);   // refill the slot consumed in step t-1
            float acc[3][R];
            f32x2 pacc[3][R];                     // (even k, odd k) partial sums of each dot product, packed
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int rr = 0; rr < R; ++rr) pacc[g][rr] = 0ull;
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int rr = 0; rr < R; ++rr) {
                    const ulonglong2 hv = *reinterpret_cast<const ulonglong2*>(&hs[cur][rr][4 * (2 * i + ks)]);
#pragma unroll
                    for (int g = 0; g < 3; ++g) {
                        pacc[g][rr] = ffma2(w[g][2 * i], hv.x, pacc[g][rr]);
                        pacc[g][rr] = ffma2(w[g][2 * i + 1], hv.y, pacc[g][rr]);
                    }
                }
            GRU_STAMP(2);
            if (kLateIssue) issue(t + kGiDepth - 1);
            GRU_STAMP(3);
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int rr = 0; rr < R; ++rr) {
                    float ev, od;
                    unpack2(pacc[g][rr], ev, od);
                    acc[g][rr] = ev + od;
                    acc[g][rr] += __shfl_xor_sync(0xffffffffu, acc[g][rr], 1);
                }
            GRU_STAMP(4);
            const float* gring = &ring[t % kGiDepth][0][0];
#pragma unroll
            for (int q = 0; q < OWN; ++q) {
                const int e = 2 * q, o = (2 * q + 1 < R) ? 2 * q + 1 : 2 * q;      // static register indices
                const float ar = ks ? acc[0][o] : acc[0][e];
                const float az = ks ? acc[1][o] : acc[1][e];
                const float an = ks ? acc[2][o] : acc[2][e];
                if (own[q]) {
                    const int rr = ks + 2 * q;
                    // GRUCell (aten gru_cell): r,z = sigmoid(gi + gh); n = tanh(gi_n + r * gh_n); h' = (h - n) z + n
                    const float* gp = gring + rr * MARL_G;
                    const float gh_n = an + bh_n;
                    const float r = gate_sigmoid((ar + bh_r) + gp[j]);
                    const float z = gate_sigmoid((az + bh_z) + gp[MARL_H + j]);
                    const float n = gate_tanh(fmaf(r, gh_n, gp[2 * MARL_H + j]));
                    const float hold = hs[cur][rr][j];
                    const float hnew = fmaf(hold - n, z, n);
                    hs[cur ^ 1][rr][j] = hnew;
                    *hp[q] = hnew;
                    if (gp_out[q]) {
                        float* go = gp_out[q];
                        go[0] = r; go[MARL_H] = z; go[2 * MARL_H] = n; go[3 * MARL_H] = gh_n;
                    }
                }
                hp[q] += hstep;
                if (gp_out[q]) gp_out[q] += gstep;
            }
            cur ^= 1;
            GRU_STAMP(5);
        }
#ifdef MARL_GRU_TRACE
        if (trace && sg == a.chain_start[chain]) {
#pragma unroll
            for (int k = 0; k < 48; ++k) { trace[2 * k] = (k % 6) + 100 * (8 + k / 6); trace[2 * k + 1] = stamp[k]; }
            trace[510] = 48;
        }
#endif
        cp_async_wait<0>();
        group_sync(bar_id);
        if (S.h_last) {
#pragma unroll
            for (int q = 0; q < OWN; ++q)
                if (own[q]) S.h_last[(long long)row_at(ks + 2 * q) * MARL_H + j] = hs[cur][ks + 2 * q][j];
        }
    }
}

// This CTA's share of a chain's rows: rows are dealt out as evenly as possible over the CTAs (one CTA per SM);
// odd chains deal the remainder from the other end, so that an SM that got an extra row of the long eval
// chain does not also get an extra row of the target chain.
__device__ __forceinline__ void cta_rows(int rows, int chain, int& begin, int& count) {
    const int n = gridDim.x, base = rows / n, rem = rows % n;
    const int pos = (chain & 1) ? n - 1 - (int)blockIdx.x : (int)blockIdx.x;
    count = base + (pos < rem ? 1 : 0);
    begin = pos * base + (pos < rem ? pos : rem);
}

// Separated networks (agent-major positions): one contiguous group of CTAs per agent, each agent's B rows dealt evenly over its
// group, so that no CTA holds rows of two agents; with more agents than CTAs the plain deal (passes split by gru_pass_rows)
__device__ __forceinline__ void cta_rows_by_agent(int B, int N, int& begin, int& count) {
    const int per = (int)gridDim.x / N;
    if (per == 0) { cta_rows(B * N, 0, begin, count); return; }
    const int n = (int)blockIdx.x / per, i = (int)blockIdx.x % per;
    if (n >= N) { begin = 0; count = 0; return; }
    const int base = B / per, rem = B % per;
    count = base + (i < rem ? 1 : 0);
    begin = n * B + i * base + (i < rem ? i : rem);
}

#ifndef MARL_GRU_SPARE_SMS
#define MARL_GRU_SPARE_SMS 16
#endif
constexpr int kGruFwdSpareSMs = MARL_GRU_SPARE_SMS;
constexpr size_t gru_fwd_smem(int R) { return (size_t)(2 * R * MARL_H + kGiDepth * R * MARL_G) * sizeof(float); }

template <bool SEP>
__global__ void __launch_bounds__(kGruThreads * kGruGroups) gru_unroll_fwd_kernel(GruFwdArgs a) {
    pdl_enter();
    extern __shared__ __align__(16) float gru_smem[];
    const int grp = threadIdx.x >> 7;
    const int chain = blockIdx.y * kGruGroups + grp;
    if (chain >= a.n_chains) return;
    float* smem = gru_smem + grp * (gru_fwd_smem(kGruMaxRows) / sizeof(float));
    int begin = 0;
    for (int i = 0; i < (int)blockIdx.x; ++i) begin += a.rows_of[chain][i];
    const int count = a.rows_of[chain][blockIdx.x];
    for (int off = 0, n = 0; off < count; off += SEP ? n : kGruMaxRows) {
        n = gru_pass_rows<SEP>(begin + off, count - off, a.B);
        if (n == 1) gru_chain_fwd<1, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else if (n == 2) gru_chain_fwd<2, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else if (n <= 4) gru_chain_fwd<4, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else gru_chain_fwd<8, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        group_sync(1 + grp);
    }
}

struct GruBwdArgs {
    const float* gates;    // [B,L,N,4H]
    const float* hidden;   // [B,L,N,H]
    const float* dh_ext;   // [B,L,N,H] or null
    const float* dh_ext2;  // [B,L,N,H] or null (external dL/dhidden)
    const float* w_hh;     // [3H,H]
    const float* h0;       // [B*N,H] or null (zeros)
    float* dgi;            // [B,L,N,3H]
    float* dgh;            // [B,L,N,3H]
    float* dh0;            // [B*N,H] or null
    int B, L, N;
    const int* ep_len;     // [B] or null: a row's chain starts at its episode's last real step
    const int* row_order;  // [B*N] or null: logical position -> row (row_order_kernel)
    int agent_stride;      // separated networks (SEP instantiation): floats from agent n's W_hh to n+1's
};

constexpr int kBwdSlot = 7 * MARL_H;     // r, z, n, gh_n (4H) | h_prev | dh_ext | dh_ext2   per row and time step
constexpr int bwd_depth(int R) { return R >= 8 ? 3 : MARL_BWD_DEPTH; }
constexpr size_t gru_bwd_smem(int R) { return (size_t)(2 * R * MARL_G + bwd_depth(R) * R * kBwdSlot) * sizeof(float); }

template <int R, bool SEP>
__device__ __forceinline__ void gru_rows_bwd(const GruBwdArgs& a, int row0, int nrows, float* gru_smem) {
    constexpr int D = bwd_depth(R);
    float (*sg)[R][MARL_G] = reinterpret_cast<float (*)[R][MARL_G]>(gru_smem);                       // [2][R][3H]
    float (*ring)[R][kBwdSlot] = reinterpret_cast<float (*)[R][kBwdSlot]>(gru_smem + 2 * R * MARL_G); // [D][R][7H]
    const int tid = threadIdx.x, ks = tid & 1, j = tid >> 1;
    const int L = a.L, N = a.N;
    __shared__ int srow[kGruMaxRows];         // (the previous pass ended with a block barrier)
    if (tid < R) srow[tid] = (a.row_order && tid < nrows) ? __ldg(a.row_order + row0 + tid) : gru_position_row<SEP>(row0 + tid, a.B, N);
    __syncthreads();
    auto row_at = [&](int rr) { return srow[rr]; };
    constexpr int OWN = (R + 1) / 2;
    bool own[OWN]; long long base[OWN]; float dh_carry[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int rr = ks + 2 * q, row = row_at(rr);
        own[q] = rr < nrows;
        base[q] = own[q] ? ((long long)(row / N) * L * N + (row % N)) : 0;
        dh_carry[q] = 0.0f;
    }
    // column j of W_hh, rows m = 4*(2i+ks)+c, i = 0..23:  dh_prev[j] = dh z + sum_m dgh[m] W_hh[m, j]
    const float* w_hh = a.w_hh + (SEP ? (long long)(row0 / a.B) * a.agent_stride : 0);      // this pass's agent
    f32x2 wt[48];                                          // (rows m, m+1) pairs
#pragma unroll
    for (int i = 0; i < 24; ++i)
#pragma unroll
        for (int c = 0; c < 2; ++c)
            wt[2 * i + c] = pack2(__ldg(w_hh + (long long)(4 * (2 * i + ks) + 2 * c) * MARL_H + j),
                                  __ldg(w_hh + (long long)(4 * (2 * i + ks) + 2 * c + 1) * MARL_H + j));
    // cp.async work list: per row 112 chunks of 16 B (64 gates, 16 h_prev, 16 dh_ext, 16 dh_ext2); the
    // per-chunk source pointer at t = 0 and its per-step stride are fixed, so they are computed once.
    constexpr int NCH = (R * 112 + kGruThreads - 1) / kGruThreads;
    const float* csrc[NCH]; int cstride[NCH], cdst[NCH], ckind[NCH];
#pragma unroll
    for (int l = 0; l < NCH; ++l) {
        const int c = tid + l * kGruThreads, rr = c / 112, ch = c % 112, row = row_at(rr);
        csrc[l] = nullptr; cstride[l] = 0; cdst[l] = rr * kBwdSlot + ch * 4; ckind[l] = 0;
        if (c < R * 112 && rr < nrows) {
            const long long idx0 = (long long)(row / N) * L * N + (row % N);
            if (ch < 64) { csrc[l] = a.gates + idx0 * (4 * MARL_H) + ch * 4; cstride[l] = N * 4 * MARL_H; }
            else if (ch < 80) { csrc[l] = a.hidden + (idx0 - N) * MARL_H + (ch - 64) * 4; cstride[l] = N * MARL_H; ckind[l] = 1;
                                 if (a.h0) ckind[l] = 2; }
            else if (ch < 96) { if (a.dh_ext) { csrc[l] = a.dh_ext + idx0 * MARL_H + (ch - 80) * 4; cstride[l] = N * MARL_H; } }
            else { if (a.dh_ext2) { csrc[l] = a.dh_ext2 + idx0 * MARL_H + (ch - 96) * 4; cstride[l] = N * MARL_H; } }
        }
    }
    auto issue = [&](int t) {
        if (t >= 0) {
            float* slot = &ring[t % D][0][0];
#pragma unroll
            for (int l = 0; l < NCH; ++l) {
                if (!csrc[l]) continue;
                if (ckind[l] != 0 && t == 0) {      // h_prev of the first step: h0 (or zeros, handled by the consumer)
                    if (ckind[l] == 2) cp_async16(slot + cdst[l], a.h0 + (long long)row_at(cdst[l] / kBwdSlot) * MARL_H + (cdst[l] % kBwdSlot - 4 * MARL_H));
                    continue;
                }
                cp_async16(slot + cdst[l], csrc[l] + (long long)t * cstride[l]);
            }
        }
        cp_async_commit();
    };
    for (int idx = tid; idx < 2 * R * MARL_G; idx += kGruThreads) (&sg[0][0][0])[idx] = 0.0f;
    // per-step output pointers of the rows this lane owns, walked backwards one time step (N rows) per iteration
    float* pi_[OWN]; float* ph_[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        pi_[q] = a.dgi + (base[q] + (long long)(L - 1) * N) * MARL_G + j;
        ph_[q] = a.dgh + (base[q] + (long long)(L - 1) * N) * MARL_G + j;
    }
    const long long ostep = (long long)N * MARL_G;
    // early exit (SURVEY 8(f) N3): behind the longest episode of this pass every upstream gradient is masked to zero, so the
    // chain would only produce zeros there -- they are written directly and the chain starts at that episode's last step
    int Lp = L;
    if (a.ep_len) {
        Lp = 1;
        for (int rr = 0; rr < nrows; ++rr) Lp = max(Lp, min(L, __ldg(a.ep_len + row_at(rr) / N)));
        const int tail = L - Lp;
        for (int idx = tid; idx < tail * nrows * (MARL_G / 4); idx += kGruThreads) {
            const int c4 = idx % (MARL_G / 4), rr = (idx / (MARL_G / 4)) % nrows, t = Lp + idx / ((MARL_G / 4) * nrows);
            const int row = row_at(rr);
            const long long off = (((long long)(row / N) * L + t) * N + (row % N)) * MARL_G + 4 * c4;
            *reinterpret_cast<float4*>(a.dgi + off) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(a.dgh + off) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int q = 0; q < OWN; ++q) { pi_[q] -= (long long)tail * ostep; ph_[q] -= (long long)tail * ostep; }
    }
#pragma unroll
    for (int d = 0; d < D - 1; ++d) issue(Lp - 1 - d);
    cp_async_wait<D - 2>();
    __syncthreads();
    int cur = 0;
    for (int t = Lp - 1; t >= 0; --t) {
        float dh_dir[OWN];
#pragma unroll
        for (int q = 0; q < OWN; ++q) {
            dh_dir[q] = 0.0f;
            if (own[q]) {
                const int rr = ks + 2 * q;
                const float* sl = &ring[t % D][rr][0];
                const float g_r = sl[j], g_z = sl[MARL_H + j], g_n = sl[2 * MARL_H + j], g_hn = sl[3 * MARL_H + j];
                const float hprev = (t > 0 || a.h0) ? sl[4 * MARL_H + j] : 0.0f;
                float dh = dh_carry[q];
                if (a.dh_ext) dh += sl[5 * MARL_H + j];
                if (a.dh_ext2) dh += sl[6 * MARL_H + j];
                // h' = (h - n) z + n ; n = tanh(gi_n + r (W_hn h + b_hn)) ; r, z = sigmoid(gi + gh)
                const float dn_pre = dh * (1.0f - g_z) * (1.0f - g_n * g_n);
                const float dz_pre = dh * (hprev - g_n) * g_z * (1.0f - g_z);
                const float dr_pre = dn_pre * g_hn * g_r * (1.0f - g_r);
                const float dghn = dn_pre * g_r;
                dh_dir[q] = dh * g_z;
                float* pi = pi_[q];
                float* ph = ph_[q];
                pi[0] = dr_pre; pi[MARL_H] = dz_pre; pi[2 * MARL_H] = dn_pre;
                ph[0] = dr_pre; ph[MARL_H] = dz_pre; ph[2 * MARL_H] = dghn;
                sg[cur][rr][j] = dr_pre; sg[cur][rr][MARL_H + j] = dz_pre; sg[cur][rr][2 * MARL_H + j] = dghn;
            }
            pi_[q] -= ostep; ph_[q] -= ostep;
        }
        // the refill of the slot of step t+1 (consumed before the previous barrier): early when many rows keep the CTA
        // throughput-bound, behind the FMAs (see the forward kernel) when the chain is latency-bound
        constexpr bool kLateIssue = R <= 2;
        if (!kLateIssue) { issue(t - (D - 1)); cp_async_wait<D - 2>(); }
        else cp_async_wait<D - 3>();     // only D-2 groups are pending here: step t-1 has landed
        __syncthreads();                 // dgh of step t visible; ring[t-1] visible
        float part[R];
        f32x2 pab[R], pcd[R];                   // four partial sums per row in two packed accumulators: short dependent chains
#pragma unroll
        for (int rr = 0; rr < R; ++rr) { pab[rr] = 0ull; pcd[rr] = 0ull; }
#pragma unroll
        for (int i = 0; i < 24; ++i)
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&sg[cur][rr][4 * (2 * i + ks)]);
                pab[rr] = ffma2(wt[2 * i], v.x, pab[rr]);
                pcd[rr] = ffma2(wt[2 * i + 1], v.y, pcd[rr]);
            }
        if (kLateIssue) issue(t - (D - 1));
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            float pa, pb, pc, pd;
            unpack2(pab[rr], pa, pb); unpack2(pcd[rr], pc, pd);
            part[rr] = (pa + pb) + (pc + pd);
            part[rr] += __shfl_xor_sync(0xffffffffu, part[rr], 1);
        }
#pragma unroll
        for (int q = 0; q < OWN; ++q) {
            const int e = 2 * q, o = (2 * q + 1 < R) ? 2 * q + 1 : 2 * q;
            dh_carry[q] = dh_dir[q] + (ks ? part[o] : part[e]);
        }
        cur ^= 1;
    }
    cp_async_wait<0>();
    if (a.dh0) {
#pragma unroll
        for (int q = 0; q < OWN; ++q)
            if (own[q]) a.dh0[(long long)row_at(ks + 2 * q) * MARL_H + j] = dh_carry[q];
    }
    __syncthreads();
}

#ifndef MARL_GRU_BWD_CTAS
#define MARL_GRU_BWD_CTAS 2
#endif
constexpr int kGruBwdCtasPerSm = MARL_GRU_BWD_CTAS;      // 254 registers x 128 threads and ~55 KB of shared memory: two CTAs fit an SM
// up to two rows per SM: one CTA per row (see marl_agent_unroll_bwd)
static int gru_bwd_ctas(int rows) { return rows <= kGruBwdCtasPerSm * kNumSMs ? rows : kNumSMs; }
constexpr size_t gru_bwd_smem_max() { return gru_bwd_smem(8) > gru_bwd_smem(4) ? gru_bwd_smem(8) : gru_bwd_smem(4); }

template <bool SEP>
__global__ void __launch_bounds__(kGruThreads) gru_unroll_bwd_kernel(GruBwdArgs a) {
    pdl_enter();
    extern __shared__ __align__(16) float gru_smem[];
    int begin, count;
    if (SEP) cta_rows_by_agent(a.B, a.N, begin, count);
    else cta_rows(a.B * a.N, 0, begin, count);
    for (int off = 0, n = 0; off < count; off += SEP ? n : kGruMaxRows) {
        n = gru_pass_rows<SEP>(begin + off, count - off, a.B);
        if (n == 1) gru_rows_bwd<1, SEP>(a, begin + off, n, gru_smem);
        else if (n == 2) gru_rows_bwd<2, SEP>(a, begin + off, n, gru_smem);
        else if (n <= 4) gru_rows_bwd<4, SEP>(a, begin + off, n, gru_smem);
        else gru_rows_bwd<8, SEP>(a, begin + off, n, gru_smem);
    }
}

// Rows of every chain per CTA.  The kernel ends when its slowest CTA does, and a CTA's time is roughly
// (steps of the chain) x (rows it advances), so rows are dealt by water-filling on that weighted load: the first
// chain evenly, every further chain onto the CTAs that carry the least so far.  At cfg 2 (160 rows, 148 CTAs) the 12
// CTAs with two rows of the 240-step eval chain get no row of the 120-step target chain.
// Separated networks (`agents` > 1): the CTAs form one contiguous group per agent (n_ctas / agents each, the rest idle) and
// each agent's B rows are water-filled onto its own group, so that no CTA's range -- and no pass -- holds rows of two agents.
// (With more agents than CTAs the plain deal is kept and the kernel splits a pass at an agent boundary, gru_pass_rows.)
static void water_fill(const double* load, int c0, int c1, int rows, double w, int* cnt) {
    // water level by bisection: CTA i takes floor((level - load_i) / w) rows
    double lo = 0.0, hi = 0.0;
    for (int i = c0; i < c1; ++i) hi = load[i] > hi ? load[i] : hi;
    hi += w * (rows / (c1 - c0) + 2);
    for (int it = 0; it < 60; ++it) {
        const double mid = 0.5 * (lo + hi);
        long long tot = 0;
        for (int i = c0; i < c1; ++i) tot += mid > load[i] ? (long long)((mid - load[i]) / w) : 0;
        if (tot >= rows) hi = mid; else lo = mid;
    }
    int tot = 0;
    for (int i = c0; i < c1; ++i) { cnt[i] = lo > load[i] ? (int)((lo - load[i]) / w) : 0; tot += cnt[i]; }
    while (tot < rows) {                       // the remainder goes, one row each, to the least loaded CTAs
        int best = c0;
        for (int i = c0 + 1; i < c1; ++i)
            if (load[i] + w * cnt[i] < load[best] + w * cnt[best]) best = i;
        ++cnt[best]; ++tot;
    }
    while (tot > rows) {                       // (bisection overshoot: take back from the most loaded)
        int worst = -1;
        for (int i = c0; i < c1; ++i)
            if (cnt[i] > 0 && (worst < 0 || load[i] + w * cnt[i] > load[worst] + w * cnt[worst])) worst = i;
        --cnt[worst]; --tot;
    }
}

static void plan_rows(GruFwdArgs& ga, int rows, int n_ctas, int agents) {
    double load[kNumSMs] = {};
    const int per = agents > 1 ? n_ctas / agents : 0;      // CTAs per agent group (0: one group of all CTAs)
    for (int c = 0; c < ga.n_chains; ++c) {
        const double w = (double)ga.chain_len[c];
        int cnt[kNumSMs] = {};
        if (per > 0)
            for (int g = 0; g < agents; ++g) water_fill(load, g * per, (g + 1) * per, rows / agents, w, cnt);
        else
            water_fill(load, 0, n_ctas, rows, w, cnt);
        for (int i = 0; i < n_ctas; ++i) { ga.rows_of[c][i] = (unsigned short)cnt[i]; load[i] += w * cnt[i]; }
    }
}

// ---- length-sorted row deal (SURVEY 8(f) N3) ------------------------------------------------------------------------------
// With per-episode early exit a CTA's time is (steps of its rows) x (cost of a step at its row count), and rows that share a
// pass advance in lock-step to the longest of them.  The plans above fix HOW MANY rows each CTA takes; this kernel decides
// WHICH: rows are ranked by episode length (longest first, ties by index: the agents of an episode stay together) and dealt pass
// by pass -- the first pass (up to 8 rows) of every CTA, then the second, ... -- within a pass level to the CTAs in the order
// `seq` (fewest rows first: at config 2 the 28 CTAs that carry two rows of the 240-step chain get the 56 shortest rows), the
// direction alternating from level to level so that the sums stay balanced.  out[logical position] = row.
constexpr int kMaxOrderCtas = 2 * kNumSMs;      // the BPTT kernel runs up to two one-row CTAs per SM
constexpr int kMaxOrderEpisodes = 1024;          // (larger batches keep the index order: the ranking below is O(B^2 / 256) per block)
constexpr int kOrderWarps = 8;
template <int C>
struct OrderPlan {
    int n_ctas;                 // 0: unused
    int* out;                   // [B*N]
    const int* ep_len;          // [B]
    unsigned short cnt[C];      // rows of CTA c (its logical positions are contiguous, CTA after CTA)
    unsigned short pos[C];      // place of CTA c in the deal: 0 gets the longest rows of a pass level, n_ctas - 1 the shortest
};
struct OrderArgs {
    OrderPlan<kNumSMs> fwd[kMaxStreams];
    OrderPlan<kMaxOrderCtas> bwd;
    int B, N;
};

// grid (ceil(n_ctas / 8), plans), one warp per CTA of the plan
__global__ void __launch_bounds__(kOrderWarps * 32) row_order_kernel(const __grid_constant__ OrderArgs a) {
    pdl_enter();
    __shared__ unsigned short cnt[kMaxOrderCtas], pos[kMaxOrderCtas];
    __shared__ unsigned short ep_of_rank[kMaxOrderEpisodes];
    __shared__ int s_n;
    const int k = blockIdx.y;
    int* out; const int* ep_len;
    if (k < kMaxStreams) {
        out = a.fwd[k].out; ep_len = a.fwd[k].ep_len;
        if (threadIdx.x == 0) s_n = a.fwd[k].n_ctas;
        for (int i = threadIdx.x; i < kNumSMs; i += blockDim.x) { cnt[i] = a.fwd[k].cnt[i]; pos[i] = a.fwd[k].pos[i]; }
    } else {
        out = a.bwd.out; ep_len = a.bwd.ep_len;
        if (threadIdx.x == 0) s_n = a.bwd.n_ctas;
        for (int i = threadIdx.x; i < kMaxOrderCtas; i += blockDim.x) { cnt[i] = a.bwd.cnt[i]; pos[i] = a.bwd.pos[i]; }
    }
    __syncthreads();
    const int n_ctas = s_n, B = a.B, N = a.N;
    if (n_ctas == 0 || (int)blockIdx.x * kOrderWarps >= n_ctas) return;
    // rank of every episode: the episodes in front of b are the longer ones and the equally long earlier ones
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const int len = __ldg(ep_len + b);
        int rank = 0;
        for (int o = 0; o < B; ++o) { const int lo = __ldg(ep_len + o); rank += (lo > len || (lo == len && o < b)) ? 1 : 0; }
        ep_of_rank[rank] = (unsigned short)b;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, c = blockIdx.x * kOrderWarps + (threadIdx.x >> 5);
    if (c >= n_ctas) return;
    const int mine = cnt[c], mypos = pos[c];
    int begin = 0;                                  // logical position of this CTA's first row
    for (int o = lane; o < c; o += 32) begin += cnt[o];
    begin = (int)warp_sum((float)begin);            // (exact: < 2^24 rows)
    int level_start = 0;                            // sorted position of the first row of pass level p
    for (int p = 0; p * kGruMaxRows < mine; ++p) {
        int before = 0, width = 0;                  // rows of level p dealt before this CTA's / in the whole level
        for (int o = lane; o < n_ctas; o += 32) {
            const int w = min(max((int)cnt[o] - kGruMaxRows * p, 0), kGruMaxRows);
            width += w;
            if ((p & 1) ? pos[o] > mypos : pos[o] < mypos) before += w;        // the deal runs backwards on odd levels
        }
        before = (int)warp_sum((float)before); width = (int)warp_sum((float)width);
        const int w = min(mine - kGruMaxRows * p, kGruMaxRows);
        if (lane < w) {
            const int sorted = level_start + before + lane;
            out[begin + kGruMaxRows * p + lane] = (int)ep_of_rank[sorted / N] * N + sorted % N;
        }
        level_start += width;
    }
}

// pos = place of every CTA when the CTAs are sorted by (rows, index) ascending.  BPTT with one-row CTAs and more CTAs than SMs: the
// CTAs that have an SM to themselves come first, the ones that share one (i and i + kNumSMs, as the block scheduler places them) last
template <int C>
static void order_plan_fill(OrderPlan<C>& pl, const unsigned short* cnt, int n_ctas, const int* ep_len, int* out) {
    pl.n_ctas = n_ctas; pl.out = out; pl.ep_len = ep_len;
    unsigned short seq[C];
    for (int c = 0; c < C; ++c) { pl.cnt[c] = c < n_ctas ? cnt[c] : 0; pl.pos[c] = 0; }
    int m = 0;
    unsigned short mx = 0;
    for (int c = 0; c < n_ctas; ++c) mx = cnt[c] > mx ? cnt[c] : mx;
    const int shared = (mx <= 1 && n_ctas > kNumSMs) ? n_ctas - kNumSMs : 0;
    if (shared) {
        for (int c = shared; c < kNumSMs; ++c) seq[m++] = (unsigned short)c;
        for (int c = 0; c < shared; ++c) { seq[m++] = (unsigned short)c; seq[m++] = (unsigned short)(c + kNumSMs); }
    } else {
        for (int c = 0; c < n_ctas; ++c) seq[m++] = (unsigned short)c;
        std::stable_sort(seq, seq + n_ctas, [&](unsigned short x, unsigned short y) { return cnt[x] < cnt[y]; });
    }
    for (int i = 0; i < n_ctas; ++i) pl.pos[seq[i]] = (unsigned short)i;
}

// (O may be 0 or negative for a FULL input, where only O + A + N = the network's input width is meaningful; the entry points
// check O > 0 for the composed [obs | last_action | agent_id] input)
// ep_len[b] = 1 + last step with padded == 0 (one warp per episode)
__global__ void __launch_bounds__(256) episode_lengths_kernel(const float* padded, int B, int L, int* ep_len) {
    pdl_enter();
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    int last = 0;
    for (int t = lane; t < L; t += 32)
        if (padded[(long long)b * L + t] == 0.f) last = t + 1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    if (lane == 0) ep_len[b] = max(last, 1);
}

static int check_dims(const marl_dims* d) {
    if (!d || d->B <= 0 || d->L <= 0 || d->N <= 0 || d->A <= 0 || d->O + d->A + d->N <= 0 || d->S < 0) return MARL_EINVAL;
    return MARL_OK;
}

// Separated networks: the rows of agent z = blockIdx.z of a launch batched over the agents, row m = b*L + t of problem z being
// row (b, t, z): [obs | last action (one step back within the episode when shifted) if last_action | eye(N)[z] if agent_id]
static LinOperand separated_input(const marl_dims* d, const float* obs, const float* onehot, int shift, int last_action, int agent_id) {
    LinOperand in = plain_operand(obs, d->N * d->O, d->O, d->O);
    if (last_action) {
        in.x2 = onehot; in.ldx2 = d->N * d->A; in.K2 = d->A; in.x2_bs = d->A;
        in.x2_shift = shift ? 1 : 0; in.x2_period = d->L;
    }
    if (agent_id) { in.onehot_mod = d->N; in.onehot_z = 1; }
    return in;
}

// The input blocks a stream reads: separated networks and shared streams that opt in (input_flags) select them with
// last_action / agent_id; any other shared stream reads all three, whatever those fields hold
struct InputBlocks { int last_action, agent_id; };
static InputBlocks input_blocks(int stride, int input_flags, int last_action, int agent_id) {
    if (stride || input_flags) return InputBlocks{last_action ? 1 : 0, agent_id ? 1 : 0};
    return InputBlocks{1, 1};
}

// the input width of the network: O + A*last_action + N*agent_id (a full input row is as wide as the composed one)
static int agent_input_width(const marl_dims* d, InputBlocks f) {
    return d->O + (f.last_action ? d->A : 0) + (f.agent_id ? d->N : 0);
}

// A layer of the agent: one problem over all rows (shared), or one launch batched over the agents (separated: problem z is
// agent z's B*L rows, N rows apart, with agent z's weights `stride` floats behind agent 0's)
static LinearFwd agent_layer(const marl_dims* d, const LinOperand& in, const float* w, int ldw, const float* b, float* y, int width, int stride) {
    LinearFwd f{};
    f.in = in; f.w = w; f.ldw = ldw; f.bias = b; f.y = y; f.N = width;
    if (stride) { f.M = d->B * d->L; f.batch = d->N; f.w_bs = stride; f.b_bs = stride; f.ldy = d->N * width; f.y_bs = width; }
    else { f.M = d->B * d->L * d->N; f.batch = 1; f.ldy = width; }
    return f;
}

// Shared network: row m = (b*L + t)*N + n is [obs | last action (N rows back when shifted) if present | eye(N)[n] if present]
static LinOperand agent_input(const marl_dims* d, const float* obs, const float* onehot, int shift, int full, InputBlocks f) {
    if (full) return plain_operand(obs, d->O + d->A + d->N, d->O + d->A + d->N);
    LinOperand in{};
    in.x = obs; in.ldx = d->O; in.K1 = d->O; in.x_bs = 0;
    if (f.last_action) {
        in.x2 = onehot; in.ldx2 = d->A; in.K2 = d->A; in.x2_bs = 0;
        in.x2_shift = shift ? d->N : 0;
        in.x2_period = d->L * d->N;
    }
    in.onehot_mod = f.agent_id ? d->N : 0;
    return in;
}

}  // namespace marl

using namespace marl;

extern "C" int marl_episode_lengths(const float* padded, int B, int L, int* ep_len, void* stream) {
    if (!padded || !ep_len || B <= 0 || L <= 0) return MARL_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    { ProfScope ps_("episode_lengths_kernel", st); launch_pdl(episode_lengths_kernel, dim3((B + 7) / 8), dim3(256), 0, st, padded, B, L, ep_len); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

extern "C" int marl_agent_unroll_fwd(const marl_dims* d, const marl_unroll_stream* s, int n_streams, void* stream) {
    if (check_dims(d) || !s || n_streams < 1 || n_streams > kMaxStreams) return MARL_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    pdl_scope((long long)d->B * d->L * d->N);
    const int rows_total = d->B * d->L * d->N;
    // separated networks: one stride for the call, no full input, no W_ih^T (batch 1 only), no early exit
    const int stride = s[0].agent_stride;
    const bool sep = stride != 0;
    auto blocks = [&](int i) { return input_blocks(stride, s[i].input_flags, s[i].last_action, s[i].agent_id); };
    for (int i = 0; i < n_streams; ++i) {
        const marl_unroll_stream& u = s[i];
        if (u.agent_stride != stride || stride < 0 || (stride & 3)) return MARL_EINVAL;
        if (sep && (u.full_input || u.w_ih_t || u.ep_len || u.padded || u.row_order || u.row_order_bwd)) return MARL_EINVAL;
        if (!sep && u.input_flags && u.full_input) return MARL_EINVAL;
        const bool need_onehot = !u.full_input && blocks(i).last_action;
        if (!s[i].obs || (need_onehot && !s[i].onehot) || !s[i].hidden || !s[i].x || !s[i].gi) return MARL_EINVAL;
        if (!s[i].full_input && d->O <= 0) return MARL_EINVAL;
        if (s[i].h0_from >= i) return MARL_EINVAL;
        if (s[i].h0_from >= 0 && s[s[i].h0_from].ep_len) return MARL_EINVAL;     // a continued stream must run to L (header)
    }
    // phase B: build chains (a stream whose h0_from == j continues chain of j; j must be a chain tail)
    const int I = agent_input_width(d, blocks(0));
    for (int i = 0; i < n_streams; ++i)
        if (agent_input_width(d, blocks(i)) != I) return MARL_EINVAL;
    GruFwdArgs ga{};
    ga.B = d->B; ga.L = d->L; ga.N = d->N; ga.agent_stride = stride;
    int order[kMaxStreams], n_ordered = 0;
    bool used[kMaxStreams] = {};
    for (int i = 0; i < n_streams; ++i) {
        if (s[i].h0_from >= 0) continue;
        int c = ga.n_chains++;
        ga.chain_start[c] = n_ordered;
        ga.h0[c] = s[i].h0;
        int cur = i;
        while (cur >= 0) {
            order[n_ordered++] = cur; used[cur] = true;
            int nxt = -1;
            for (int k = cur + 1; k < n_streams; ++k)
                if (!used[k] && s[k].h0_from == cur) { nxt = k; break; }
            cur = nxt;
        }
        ga.chain_len[c] = n_ordered - ga.chain_start[c];
    }
    if (n_ordered != n_streams) return MARL_EINVAL;   // two successors of one stream are not supported
    for (int k = 0; k < n_streams; ++k) {
        const marl_unroll_stream& u = s[order[k]];
        ga.seg[k] = GruSegment{u.gi, u.params.w_hh, u.params.b_hh, u.hidden, u.gates, u.h_last, u.ep_len};
    }
    // A recurrence CTA takes an SM's whole register file, so nothing else runs beside it.  When leaving a few SMs out does not
    // add a row to the fullest CTA, they go to the kernels sibling streams have queued (the target hyper-network forward of
    // QMIX otherwise waits for this kernel to END, in front of the mixing kernel).
    // Separated networks deal each agent's B rows onto its own group of n_ctas / N CTAs (plan_rows), so the fullest CTA takes
    // ceil(B / (n_ctas / N)) rows -- at cfg 4 (N = 27, B = 32) 7 where the plain deal would give 6 but split passes at agent
    // boundaries -- and both choices below are made on that count.
    const int rows = d->B * d->N;
    auto fullest = [&](int n) { return (sep && n / d->N > 0) ? (d->B + n / d->N - 1) / (n / d->N) : (rows + n - 1) / n; };
    int n_ctas = rows < kNumSMs ? rows : kNumSMs;
    if (rows > kNumSMs && fullest(kNumSMs - kGruFwdSpareSMs) == fullest(kNumSMs)) n_ctas = kNumSMs - kGruFwdSpareSMs;
    if (fullest(n_ctas) + 2 > 65535) return MARL_EINVAL;      // rows_of is unsigned short
    plan_rows(ga, rows, n_ctas, sep ? d->N : 1);
    std::unique_ptr<ForkJoin> order_lane;
    {
        // length-sorted deal of the rows (row_order_kernel): a chain whose streams carry an episode-length array and a scratch
        // array; the order for this step's BPTT kernel (same rule on ITS plan) comes out of the same launch
        OrderArgs oa{};
        oa.B = d->B; oa.N = d->N;
        bool any = false;
        for (int c = 0; c < ga.n_chains; ++c) {
            const int* len = nullptr; int* out = nullptr;
            for (int k = ga.chain_start[c]; k < ga.chain_start[c] + ga.chain_len[c]; ++k) {
                if (!len) len = s[order[k]].ep_len;
                if (!out) out = s[order[k]].row_order;
            }
            if (!len || !out || d->B > kMaxOrderEpisodes) continue;
            order_plan_fill(oa.fwd[c], ga.rows_of[c], n_ctas, len, out);
            ga.row_order[c] = out;
            any = true;
        }
        for (int i = 0; i < n_streams && !oa.bwd.n_ctas; ++i)
            if (s[i].row_order_bwd && d->B <= kMaxOrderEpisodes) {
                const int* len = nullptr;
                for (int k = 0; k < n_streams && !len; ++k) len = s[k].ep_len;
                if (!len) return MARL_EINVAL;
                unsigned short cnt[kMaxOrderCtas];
                const int nb = gru_bwd_ctas(rows);
                for (int c = 0; c < nb; ++c) cnt[c] = (unsigned short)(rows / nb + (c < rows % nb ? 1 : 0));     // cta_rows()
                order_plan_fill(oa.bwd, cnt, nb, len, s[i].row_order_bwd);
                any = true;
            }
        // episode lengths + row orders run on a forked lane BESIDE the input layers; the recurrence waits for both
        const float* padded = nullptr; int* len_out = nullptr;
        for (int i = 0; i < n_streams && !padded; ++i)
            if (s[i].padded && s[i].ep_len) { padded = s[i].padded; len_out = const_cast<int*>(s[i].ep_len); }
        if (any || padded) {
            order_lane.reset(new ForkJoin(st, 2));
            cudaStream_t ls = order_lane->lane(1);
            if (padded) {
                ProfScope ps_("episode_lengths_kernel", ls);
                launch_pdl(episode_lengths_kernel, dim3((d->B + 7) / 8), dim3(256), 0, ls, padded, d->B, d->L, len_out);
                MARL_LAUNCH_CHECK();
            }
            if (any) {
                ProfScope ps_("row_order_kernel", ls);
                launch_pdl(row_order_kernel, dim3((gru_bwd_ctas(rows) + kOrderWarps - 1) / kOrderWarps, kMaxStreams + 1), dim3(kOrderWarps * 32), 0, ls, oa);
                MARL_LAUNCH_CHECK();
            }
        }
    }
    // phase A: x = relu(fc1(input)), gi = W_ih x + b_ih for every stream
    auto fc1_of = [&](int i) {
        const LinOperand in = sep ? separated_input(d, s[i].obs, s[i].onehot, s[i].shift_onehot, s[i].last_action, s[i].agent_id)
                                  : agent_input(d, s[i].obs, s[i].onehot, s[i].shift_onehot, s[i].full_input, blocks(i));
        LinearFwd f = agent_layer(d, in, s[i].params.fc1_w, I, s[i].params.fc1_b, s[i].x, MARL_H, stride);
        f.relu = 1;
        return f;
    };
    auto ih_of = [&](int i) {
        const LinOperand in = sep ? plain_operand(s[i].x, d->N * MARL_H, MARL_H, MARL_H) : plain_operand(s[i].x, MARL_H, MARL_H);
        return agent_layer(d, in, s[i].params.w_ih, MARL_H, s[i].params.b_ih, s[i].gi, MARL_G, stride);
    };
    bool grouped = false;
    if (!sep) {      // (the fused input-layer kernel stages one shared weight set: separated streams take the unfused path)
        // fused path (csrc/front.cu): both layers of every stream in ONE persistent launch, x handed from the first GEMM to the
        // second through tensor memory
        FrontArgs fa{};
        fa.rows = rows_total; fa.I = I;
        for (int i = 0; i < n_streams; ++i) {
            fa.s[i].in = agent_input(d, s[i].obs, s[i].onehot, s[i].shift_onehot, s[i].full_input, blocks(i));
            fa.s[i].x = s[i].x; fa.s[i].gi = s[i].gi;
            fa.s[i].store_x = s[i].gates != nullptr;
            fa.set[i].w1 = s[i].params.fc1_w; fa.set[i].b1 = s[i].params.fc1_b;
            fa.set[i].w_ih = s[i].params.w_ih; fa.set[i].b_ih = s[i].params.b_ih;
            fa.set[i].w_ih_t = s[i].w_ih_t;
        }
        if (front_plan(fa, n_streams)) {
            const int rc = front_launch(fa, n_streams, kGruPrio, st);
            if (rc) return rc;
            grouped = true;
        }
    }
    if (!grouped) {
        for (int i = 0; i < n_streams; ++i)
            if (s[i].w_ih_t) {
                const int rc = transpose_weights(s[i].params.w_ih, MARL_H, 0, MARL_G, MARL_H, s[i].w_ih_t, st);
                if (rc) return rc;
            }
    }
    if (!grouped && !sep && tgemm_enabled()) {
        // TMA path: the streams of one layer are ONE grouped launch of persistent CTAs (csrc/tgemm.cu): 2 launches
        // instead of 2 x n_streams on forked streams
        TGBuilder b1, b2;
        bool ok = true;
        for (int i = 0; i < n_streams && ok; ++i) ok = b1.add_fwd(fc1_of(i));
        for (int i = 0; i < n_streams && ok; ++i) ok = b2.add_fwd(ih_of(i));
        if (ok) {
            LinearPrio prio_(kGruPrio);
            int rc = b1.launch(st);
            if (rc) return rc;
            if ((rc = b2.launch(st))) return rc;
            grouped = true;
        }
    }
    if (!grouped) {
        // the streams are independent -> one lane each
        ForkJoin fa(st, n_streams);
        {
            LinearPrio prio_(kGruPrio);   // placed ahead of the GEMMs other streams issue at the same moment (the mixer's hyper-networks)
            for (int i = 0; i < n_streams; ++i) {
                cudaStream_t st = fa.lane(i);
                int rc = linear_fwd(fc1_of(i), st);
                if (rc) return rc;
                rc = linear_fwd(ih_of(i), st);
                if (rc) return rc;
            }
        }
        fa.join();
    }
    {
        // one CTA per SM; each CTA advances its share of every chain side by side (one 128-thread group per chain)
        ProfScope ps_("gru_unroll_fwd_kernel", st);
        const size_t sm = kGruGroups * gru_fwd_smem(kGruMaxRows);
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(gru_unroll_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
            cudaFuncSetAttribute(gru_unroll_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
            attr_set = true;
        }
        ga.trace = trace_buffer();
        if (order_lane) order_lane->join();
        dim3 grid(n_ctas, (ga.n_chains + kGruGroups - 1) / kGruGroups);
        launch_pdl_prio(kGruPrio, sep ? gru_unroll_fwd_kernel<true> : gru_unroll_fwd_kernel<false>, grid,
                        dim3(kGruThreads * kGruGroups), sm, st, ga);
    }
    MARL_LAUNCH_CHECK();
    // phase C.  (The fork / join pair stays even when a fused mixer evaluates the heads and nothing is launched here: it takes the
    // programmatic launch edge between the recurrence and the mixing kernel, whose 480 early-resident CTAs otherwise sit on the
    // SMs beside the last steps of the recurrence -- measured 333 us per step with the pair, 345-354 us without.)
    ForkJoin fc(st, n_streams);
    for (int i = 0; i < n_streams; ++i) {
        if (!s[i].q) continue;
        cudaStream_t st = fc.lane(i);
        const LinOperand in = sep ? plain_operand(s[i].hidden, d->N * MARL_H, MARL_H, MARL_H) : plain_operand(s[i].hidden, MARL_H, MARL_H);
        int rc = linear_fwd(agent_layer(d, in, s[i].params.fc2_w, MARL_H, s[i].params.fc2_b, s[i].q, d->A, stride), st);
        if (rc) return rc;
    }
    fc.join();
    return MARL_OK;
}

extern "C" int marl_agent_unroll_bwd(const marl_dims* d, const marl_unroll_bwd* a, void* stream) {
    if (check_dims(d) || !a || !a->hidden || !a->x || !a->gates || !a->dgi || !a->dgh || !a->dx) return MARL_EINVAL;
    if (a->dq && !a->dhext) return MARL_EINVAL;
    if (!a->full_input && d->O <= 0) return MARL_EINVAL;
    const int stride = a->agent_stride;
    const bool sep = stride != 0;
    if (stride < 0 || (stride & 3)) return MARL_EINVAL;
    if (sep && (a->full_input || a->w_ih_t || a->ep_len || a->row_order)) return MARL_EINVAL;
    if (!sep && a->input_flags && a->full_input) return MARL_EINVAL;
    const InputBlocks blk = input_blocks(stride, a->input_flags, a->last_action, a->agent_id);
    if (!a->full_input && blk.last_action && !a->onehot) return MARL_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    pdl_scope((long long)d->B * d->L * d->N);
    const int rows_total = d->B * d->L * d->N;
    const int I = agent_input_width(d, blk);
    // separated networks: every layer is one launch batched over the agents -- problem z holds agent z's B*L rows, which sit
    // N rows apart (row pitch x N, column offset z x width), and its weights / gradients `stride` floats behind agent 0's
    const int nb = sep ? d->N : 1, M = sep ? d->B * d->L : rows_total, rp = sep ? d->N : 1;
    auto zs = [&](int width) -> long long { return sep ? width : 0; };
    int rc;
    if (a->dq && !a->dhext_ready) {
        // q = W2 h + b2:  dh_ext = dq . W2 ;  dW2 += dq^T h ; db2 += colsum(dq)
        LinearDgrad g{};
        g.dy = a->dq; g.lddy = rp * d->A; g.dy_bs = zs(d->A); g.w = a->params.fc2_w; g.ldw = MARL_H; g.w_bs = stride; g.w_col0 = 0;
        g.dx = a->dhext; g.lddx = rp * MARL_H; g.dx_bs = zs(MARL_H); g.M = M; g.N = d->A; g.K = MARL_H; g.batch = nb;
        if ((rc = linear_dgrad(g, st))) return rc;
    }
    GruBwdArgs ga{a->gates, a->hidden, a->dq ? a->dhext : nullptr, a->dhidden, a->params.w_hh, a->h0, a->dgi, a->dgh, a->dh0,
                  d->B, d->L, d->N, a->ep_len, (a->ep_len && d->B <= kMaxOrderEpisodes) ? a->row_order : nullptr, stride};
    const int rows = d->B * d->N;
    {
        ProfScope ps_("gru_unroll_bwd_kernel", st);
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(gru_unroll_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gru_bwd_smem_max());
            cudaFuncSetAttribute(gru_unroll_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gru_bwd_smem_max());
            attr_set = true;
        }
        const bool keep_ = pdl_small_problem();
        // measured: launched programmatically the 148 recurrence CTAs come up while the producer still runs and the
        // step gets 10-27 us slower on every config; a plain launch here, PDL for its consumers
        pdl_small_problem() = false;
        // up to two rows per SM: one CTA per row -- two co-resident one-row CTAs overlap each other's latency, where one CTA with two
        // rows serialises 2 x 96 packed FMAs per thread on the dependent chain (the 12 two-row CTAs of config 2 ended the kernel)
        const int n_ctas = gru_bwd_ctas(rows);
        launch_pdl_prio(kGruPrio, sep ? gru_unroll_bwd_kernel<true> : gru_unroll_bwd_kernel<false>, dim3(n_ctas), dim3(kGruThreads),
                        gru_bwd_smem_max(), st, ga);
        pdl_small_problem() = keep_;
    }
    MARL_LAUNCH_CHECK();
    LinearWgrad w_fc2{}, w_hh{}, w_ih{}, w_fc1{}, w_h0{};
    LinearDgrad g_dx{};
    // dW2 += dq^T h ; db2 += colsum(dq)
    w_fc2.dy = a->dq; w_fc2.lddy = rp * d->A; w_fc2.dy_bs = zs(d->A); w_fc2.in = plain_operand(a->hidden, rp * MARL_H, MARL_H, zs(MARL_H));
    w_fc2.dw = a->grads.fc2_w; w_fc2.ldw = MARL_H; w_fc2.db = a->grads.fc2_b; w_fc2.M = M; w_fc2.N = d->A; w_fc2.batch = nb;
    w_fc2.dw_bs = stride; w_fc2.db_bs = stride;
    // dW_hh += dgh^T . h_{t-1} (hidden shifted by one step, zeros at t = 0) ; db_hh
    w_hh.dy = a->dgh; w_hh.lddy = rp * MARL_G; w_hh.dy_bs = zs(MARL_G);
    {
        LinOperand in{};
        in.x = nullptr; in.K1 = 0; in.x2 = a->hidden; in.ldx2 = rp * MARL_H; in.K2 = MARL_H; in.x2_bs = zs(MARL_H);
        in.x2_shift = sep ? 1 : d->N; in.x2_period = sep ? d->L : d->L * d->N; in.onehot_mod = 0;
        w_hh.in = in;
    }
    w_hh.dw = a->grads.w_hh; w_hh.ldw = MARL_H; w_hh.db = a->grads.b_hh; w_hh.M = M; w_hh.N = MARL_G; w_hh.batch = nb;
    w_hh.dw_bs = stride; w_hh.db_bs = stride;
    // the t = 0 rows see h0 instead of zeros: one [N x H] problem per episode (separated: one [B x H] problem per agent)
    w_h0.dw = a->grads.w_hh; w_h0.ldw = MARL_H; w_h0.db = nullptr; w_h0.N = MARL_G;
    if (sep) {
        w_h0.dy = a->dgh; w_h0.lddy = d->L * d->N * MARL_G; w_h0.dy_bs = MARL_G;
        w_h0.in = plain_operand(a->h0, d->N * MARL_H, MARL_H, MARL_H);
        w_h0.M = d->B; w_h0.batch = d->N; w_h0.dw_bs = stride;
    } else {
        w_h0.dy = a->dgh; w_h0.lddy = MARL_G; w_h0.dy_bs = (long long)d->L * d->N * MARL_G;
        w_h0.in = plain_operand(a->h0, MARL_H, MARL_H, (long long)d->N * MARL_H);
        w_h0.M = d->N; w_h0.batch = d->B;
    }
    // dW_ih += dgi^T . x ; db_ih
    w_ih.dy = a->dgi; w_ih.lddy = rp * MARL_G; w_ih.dy_bs = zs(MARL_G); w_ih.in = plain_operand(a->x, rp * MARL_H, MARL_H, zs(MARL_H));
    w_ih.dw = a->grads.w_ih; w_ih.ldw = MARL_H; w_ih.db = a->grads.b_ih; w_ih.M = M; w_ih.N = MARL_G; w_ih.batch = nb;
    w_ih.dw_bs = stride; w_ih.db_bs = stride;
    // dx = (dgi . W_ih) * (x > 0)
    g_dx.dy = a->dgi; g_dx.lddy = rp * MARL_G; g_dx.dy_bs = zs(MARL_G); g_dx.w = a->params.w_ih; g_dx.ldw = MARL_H; g_dx.w_bs = stride;
    g_dx.w_col0 = 0;
    g_dx.dx = a->dx; g_dx.lddx = rp * MARL_H; g_dx.dx_bs = zs(MARL_H); g_dx.relu_src = a->x; g_dx.ldrs = rp * MARL_H; g_dx.rs_bs = zs(MARL_H);
    g_dx.M = M; g_dx.N = MARL_G; g_dx.K = MARL_H; g_dx.batch = nb;
    g_dx.wt = a->w_ih_t; g_dx.ldwt = MARL_G;      // W_ih transposed by this step's forward pass (both operands then stage with 128-bit stores)
    // dW1 += dx^T . [obs | last_action | agent_id] ; db1
    w_fc1.dy = a->dx; w_fc1.lddy = rp * MARL_H; w_fc1.dy_bs = zs(MARL_H);
    w_fc1.in = sep ? separated_input(d, a->obs, a->onehot, a->shift_onehot, a->last_action, a->agent_id)
                   : agent_input(d, a->obs, a->onehot, a->shift_onehot, a->full_input, blk);
    w_fc1.dw = a->grads.fc1_w; w_fc1.ldw = I; w_fc1.db = a->grads.fc1_b; w_fc1.M = M; w_fc1.N = MARL_H; w_fc1.batch = nb;
    w_fc1.dw_bs = stride; w_fc1.db_bs = stride;

    if (!sep && tgemm_enabled()) {
        // TMA path (csrc/tgemm.cu): the data gradient and the three weight gradients that only need the BPTT's outputs are
        // ONE grouped launch, the fc1 weight gradient (needs dx) a second, and one deterministic reduce folds every
        // split partial into the flat gradient
        TGBuilder bA, bB;
        bool ok = bA.add_dgrad(g_dx) && bA.add_wgrad(w_ih) && bA.add_wgrad(w_hh);
        if (ok && a->dq) ok = bA.add_wgrad(w_fc2);
        ok = ok && bB.add_wgrad(w_fc1);
        if (ok) {
            if ((rc = bA.launch(st))) return rc;
            if ((rc = bB.launch(st))) return rc;
            bA.move_reduce_to(bB);
            if ((rc = bB.launch_reduce(st))) return rc;
            if (a->h0 && (rc = linear_wgrad(w_h0, st))) return rc;
            return MARL_OK;
        }
    }
    // the four weight gradients and the dx chain are independent: fan them out
    ForkJoin fb(st, 4);
    if (a->dq && (rc = linear_wgrad(w_fc2, fb.lane(3)))) return rc;
    if ((rc = linear_wgrad(w_hh, fb.lane(1)))) return rc;
    if (a->h0 && (rc = linear_wgrad(w_h0, fb.lane(1)))) return rc;
    if ((rc = linear_wgrad(w_ih, fb.lane(2)))) return rc;
    // (a launch priority on the dependent pair dx -> dW1, the tail's critical path, was measured: no change)
    // (also measured: this data gradient launched plainly instead of programmatically behind the BPTT kernel, +12 us; the three
    // independent weight gradients forked behind the data gradient instead of beside it, +3 us)
    if ((rc = linear_dgrad(g_dx, st))) return rc;
    if ((rc = linear_wgrad(w_fc1, st))) return rc;
    fb.join();
    return MARL_OK;
}
