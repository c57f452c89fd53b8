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
#ifndef MARL_GI_DEPTH
#define MARL_GI_DEPTH 4
#endif
#ifndef MARL_BWD_DEPTH
#define MARL_BWD_DEPTH 6
#endif
constexpr int kGiDepth = MARL_GI_DEPTH;   // cp.async ring depth (time steps) of the forward's input gates

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

// One CTA advances R rows (b,n) of one chain through all its segments.  Thread (j, ks) = (tid / KS, tid % KS) of a group owns
// hidden unit j and the reduction indices 4 (KS i + ks) + c, so every thread keeps its 3 x 32 W_hh weights in registers for the
// whole segment at every width, and the KS lanes of a unit sit side by side in one warp.
template <int H>
struct GruWidth {
    static_assert(H == 32 || H == 64 || H == 128, "rnn_hidden_dim is 32, 64 or 128");
    static constexpr int KS = H / 32;                 // lanes per hidden unit
    static constexpr int T = H * KS;                  // threads of one group (at H = 64 one warp per SM sub-partition)
    static constexpr int G = 3 * H;
    static constexpr int kGroups = T >= 512 ? 1 : 2;  // forward: chains side by side in one CTA (512 threads fill the register file)
    // rows per pass: what fits the registers without spills (at most 128 a thread in a 512-thread group; at H = 32 every lane
    // owns every row)
    static constexpr int kMaxRows = H == 32 ? 4 : H == 64 ? 8 : 2;
    static constexpr int rows(int r) { return r < kMaxRows ? r : kMaxRows; }      // a pass size of the ladder 1, 2, 4, 8, clamped
    // row slots of a pass: lane ks reads slot ks + KS q for every q < ceil(R / KS), past the pass's rows when KS > R
    static constexpr int kSlots = kMaxRows > KS ? kMaxRows : KS;
};

// named barrier of one thread group: the forward CTA hosts one group per chain, each advancing its own rows
template <int H>
__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(GruWidth<H>::T) : "memory"); }

// the KS partial sums of one hidden unit, summed over its lanes (butterfly: every lane ends with the total)
template <int KS>
__device__ __forceinline__ float lanes_sum(float v) {
#pragma unroll
    for (int o = 1; o < KS; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// v[q * KS + ks] with register indices fixed at compile time (rows past R read v[q * KS])
template <int KS, int R>
__device__ __forceinline__ float lane_pick(const float (&v)[R], int q, int ks) {
    if constexpr (KS == 2) {      // one select of two registers (the loop below schedules the H = 64 kernels differently)
        const int e = 2 * q, o = (2 * q + 1 < R) ? 2 * q + 1 : 2 * q;
        return ks ? v[o] : v[e];
    } else {
        float r = v[q * KS];
#pragma unroll
        for (int c = 1; c < KS; ++c)
            if (q * KS + c < R && ks == c) r = v[q * KS + c];
        return r;
    }
}

// Separated networks (one parameter set per agent, SEP): logical positions are dealt agent-major, position p = n*B + b is row
// b*N + n, and a pass never straddles two agents (gru_pass_rows), so the W_hh slice in registers is the pass's agent's.
template <bool SEP>
__device__ __forceinline__ int gru_position_row(int p, int B, int N) { return SEP ? (p % B) * N + p / B : p; }
template <int H, bool SEP>
__device__ __forceinline__ int gru_pass_rows(int pos, int left, int B) {
    const int n = min(GruWidth<H>::kMaxRows, left);
    return SEP ? min(n, B - pos % B) : n;
}

template <int H>
constexpr size_t gru_fwd_smem(int R) { return (size_t)(2 * R * H + kGiDepth * R * 3 * H) * sizeof(float); }

template <int H, int R, bool SEP>
__device__ __forceinline__ void gru_chain_fwd(const GruFwdArgs& a, int chain, int row0, int nrows, float* smem, int bar_id) {
    using W = GruWidth<H>;
    constexpr int KS = W::KS, T = W::T, G = W::G, CPR = G / 4;       // CPR: 16-byte chunks of gi per row and step
    float (*hs)[R][H] = reinterpret_cast<float (*)[R][H]>(smem);                              // [2][R][H]
    float (*ring)[R][G] = reinterpret_cast<float (*)[R][G]>(smem + 2 * R * H);                // [D][R][3H]
    const int tid = threadIdx.x % T, ks = tid % KS, j = tid / KS;
    const int L = a.L, N = a.N;
    // logical position (what the CTAs are dealt) -> row b*N + n: identity, or the length-sorted deal of row_order_kernel
    // (resolved once per pass into shared memory: the previous pass ended with a group barrier)
    __shared__ int srow_all[W::kGroups][W::kSlots];
    int* srow = srow_all[bar_id - 1];
    if (tid < R) {
        const int* order = a.row_order[chain];
        srow[tid] = (order && tid < nrows) ? __ldg(order + row0 + tid) : gru_position_row<SEP>(row0 + tid, a.B, N);
    }
    group_sync<H>(bar_id);
    auto row_at = [&](int rr) { return srow[rr]; };
    constexpr int OWN = (R + KS - 1) / KS;            // rows whose gate math this lane owns: rr = ks + KS q
    bool own[OWN]; long long base[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int rr = ks + KS * q, row = row_at(rr);
        own[q] = rr < nrows;
        base[q] = own[q] ? ((long long)(row / N) * L * N + (row % N)) : 0;
    }
    // cp.async work list: R rows x CPR chunks of 16 B per time step, their sources computed once -- except in a 512-thread group,
    // whose 128 registers a thread do not hold the list: it recomputes each chunk's source per step
    constexpr bool kChunkList = T < 512;
    constexpr int NCH = (R * CPR + T - 1) / T;
    long long csrc[NCH]; int cdst[NCH];
#pragma unroll
    for (int l = 0; l < (kChunkList ? NCH : 0); ++l) {
        const int c = tid + l * T, rr = c / CPR, ch = c % CPR, row = row_at(rr);
        if (c < R * CPR && rr < nrows) {
            csrc[l] = ((long long)(row / N) * L * N + (row % N)) * G + ch * 4;
            cdst[l] = rr * G + ch * 4;
        } else { csrc[l] = -1; cdst[l] = 0; }
    }
#ifdef MARL_GRU_TRACE
    long long* trace = (a.trace && tid == 0 && chain == 0 && (blockIdx.x == 0 || blockIdx.x == 100)) ? a.trace + (blockIdx.x ? 512 : 0) : nullptr;
    unsigned stamp[48] = {};
    if (trace) { trace[508] = R; trace[509] = nrows; }
#endif
    const float* h0 = a.h0[chain];
    for (int idx = tid; idx < R * H; idx += T) {
        const int rr = idx / H, jj = idx % H, row = row_at(rr);
        hs[0][rr][jj] = (h0 && rr < nrows) ? h0[(long long)row * H + jj] : 0.0f;
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
                const float4 v = __ldg(reinterpret_cast<const float4*>(w_hh + (long long)(g * H + j) * H + 4 * (KS * i + ks)));
                w[g][2 * i] = pack2(v.x, v.y); w[g][2 * i + 1] = pack2(v.z, v.w);
            }
        const float bh_r = __ldg(b_hh + j), bh_z = __ldg(b_hh + H + j), bh_n = __ldg(b_hh + 2 * H + j);
        // per-step output pointers of the rows this lane owns, advanced by one time step (N rows) per iteration; a 512-thread group
        // keeps the (b, t, n) index of each row instead (two registers a row where the pointers take four)
        float* hp[OWN]; float* gp_out[OWN]; long long idx[OWN];
#pragma unroll
        for (int q = 0; q < OWN; ++q) {
            if constexpr (kChunkList) {
                hp[q] = S.hidden + base[q] * H + j;
                gp_out[q] = S.gates ? S.gates + base[q] * (4 * H) + j : nullptr;
            } else idx[q] = base[q];
        }
        const long long hstep = (long long)N * H, gstep = (long long)N * 4 * H;
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
                if constexpr (kChunkList) {
#pragma unroll
                    for (int l = 0; l < NCH; ++l)
                        if (csrc[l] >= 0) cp_async16(&ring[t % kGiDepth][0][0] + cdst[l], S.gi + csrc[l] + (long long)t * N * G);
                } else {
                    for (int c = tid; c < nrows * CPR; c += T) {
                        const int rr = c / CPR, ch = c % CPR, row = row_at(rr);
                        cp_async16(&ring[t % kGiDepth][rr][ch * 4], S.gi + (((long long)(row / N) * L + t) * N + (row % N)) * G + ch * 4);
                    }
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int t = 0; t < kGiDepth - 1; ++t) issue(t);
        for (int t = 0; t < Lp; ++t) {
            GRU_STAMP(0);
            cp_async_wait<kGiDepth - 2>();           // this thread's copies for step t have landed
            group_sync<H>(bar_id);                   // ... the whole group's; also orders the h double buffer
            GRU_STAMP(1);
            // Few rows per CTA = latency-bound chain: the refill's address math and LSU hand-off (~150 cycles when it sat
            // here, measured with clock64) go behind the FMAs, where they overlap the FMA drain.  Many rows per CTA =
            // throughput-bound: keep the prefetch as early as possible.  (A 512-thread group issues early: the late refill's
            // registers, live beside the accumulators, do not fit its 128 a thread.)
            constexpr bool kLateIssue = R <= 2 && T < 512;
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
                    const ulonglong2 hv = *reinterpret_cast<const ulonglong2*>(&hs[cur][rr][4 * (KS * i + ks)]);
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
                    acc[g][rr] = lanes_sum<KS>(ev + od);
                }
            GRU_STAMP(4);
            const float* gring = &ring[t % kGiDepth][0][0];
#pragma unroll
            for (int q = 0; q < OWN; ++q) {
                float ar, az, an;
                if constexpr (KS == 2) {      // (written out: through lane_pick the H = 64 kernel compiles to another schedule)
                    const int e = 2 * q, o = (2 * q + 1 < R) ? 2 * q + 1 : 2 * q;      // static register indices
                    ar = ks ? acc[0][o] : acc[0][e]; az = ks ? acc[1][o] : acc[1][e]; an = ks ? acc[2][o] : acc[2][e];
                } else {
                    ar = lane_pick<KS>(acc[0], q, ks); az = lane_pick<KS>(acc[1], q, ks); an = lane_pick<KS>(acc[2], q, ks);
                }
                if (own[q]) {
                    const int rr = ks + KS * q;
                    // GRUCell (aten gru_cell): r,z = sigmoid(gi + gh); n = tanh(gi_n + r * gh_n); h' = (h - n) z + n
                    const float* gp = gring + rr * G;
                    const float gh_n = an + bh_n;
                    const float r = gate_sigmoid((ar + bh_r) + gp[j]);
                    const float z = gate_sigmoid((az + bh_z) + gp[H + j]);
                    const float n = gate_tanh(fmaf(r, gh_n, gp[2 * H + j]));
                    const float hold = hs[cur][rr][j];
                    const float hnew = fmaf(hold - n, z, n);
                    hs[cur ^ 1][rr][j] = hnew;
                    if constexpr (kChunkList) *hp[q] = hnew;
                    else S.hidden[idx[q] * H + j] = hnew;
                    if (kChunkList ? gp_out[q] != nullptr : S.gates != nullptr) {
                        float* go = kChunkList ? gp_out[q] : S.gates + idx[q] * (4 * H) + j;
                        go[0] = r; go[H] = z; go[2 * H] = n; go[3 * H] = gh_n;
                    }
                }
                if constexpr (kChunkList) {
                    hp[q] += hstep;
                    if (gp_out[q]) gp_out[q] += gstep;
                } else idx[q] += N;
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
        group_sync<H>(bar_id);
        if (S.h_last) {
#pragma unroll
            for (int q = 0; q < OWN; ++q)
                if (own[q]) S.h_last[(long long)row_at(ks + KS * q) * H + j] = hs[cur][ks + KS * q][j];
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

template <int H, bool SEP>
__global__ void __launch_bounds__(GruWidth<H>::T * GruWidth<H>::kGroups) gru_unroll_fwd_kernel(GruFwdArgs a) {
    using W = GruWidth<H>;
    pdl_enter();
    extern __shared__ __align__(16) float gru_smem[];
    const int grp = threadIdx.x / W::T;
    const int chain = blockIdx.y * W::kGroups + grp;
    if (chain >= a.n_chains) return;
    float* smem = gru_smem + grp * (gru_fwd_smem<H>(W::kMaxRows) / sizeof(float));
    int begin = 0;
    for (int i = 0; i < (int)blockIdx.x; ++i) begin += a.rows_of[chain][i];
    const int count = a.rows_of[chain][blockIdx.x];
    for (int off = 0, n = 0; off < count; off += SEP ? n : W::kMaxRows) {
        n = gru_pass_rows<H, SEP>(begin + off, count - off, a.B);
        if (n == 1) gru_chain_fwd<H, 1, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else if (W::kMaxRows == 2 || n == 2) gru_chain_fwd<H, 2, SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else if (W::kMaxRows == 4 || n <= 4) gru_chain_fwd<H, W::rows(4), SEP>(a, chain, begin + off, n, smem, 1 + grp);
        else gru_chain_fwd<H, W::rows(8), SEP>(a, chain, begin + off, n, smem, 1 + grp);
        group_sync<H>(1 + grp);
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

constexpr int bwd_depth(int R) { return R >= 8 ? 3 : MARL_BWD_DEPTH; }
// ring slot per row and time step: r, z, n, gh_n (4H) | h_prev | dh_ext | dh_ext2
template <int H>
constexpr size_t gru_bwd_smem(int R) { return (size_t)(2 * R * 3 * H + bwd_depth(R) * R * 7 * H) * sizeof(float); }

template <int H, int R, bool SEP>
__device__ __forceinline__ void gru_rows_bwd(const GruBwdArgs& a, int row0, int nrows, float* gru_smem) {
    using W = GruWidth<H>;
    constexpr int KS = W::KS, T = W::T, G = W::G, SLOT = 7 * H, CPR = SLOT / 4;   // CPR: 16-byte chunks of a slot
    constexpr int D = bwd_depth(R);
    float (*sg)[R][G] = reinterpret_cast<float (*)[R][G]>(gru_smem);                          // [2][R][3H]
    float (*ring)[R][SLOT] = reinterpret_cast<float (*)[R][SLOT]>(gru_smem + 2 * R * G);     // [D][R][7H]
    const int tid = threadIdx.x, ks = tid % KS, j = tid / KS;
    const int L = a.L, N = a.N;
    __shared__ int srow[W::kSlots];           // (the previous pass ended with a block barrier)
    if (tid < R) srow[tid] = (a.row_order && tid < nrows) ? __ldg(a.row_order + row0 + tid) : gru_position_row<SEP>(row0 + tid, a.B, N);
    __syncthreads();
    auto row_at = [&](int rr) { return srow[rr]; };
    constexpr int OWN = (R + KS - 1) / KS;
    bool own[OWN]; long long base[OWN]; float dh_carry[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int rr = ks + KS * q, row = row_at(rr);
        own[q] = rr < nrows;
        base[q] = own[q] ? ((long long)(row / N) * L * N + (row % N)) : 0;
        dh_carry[q] = 0.0f;
    }
    // column j of W_hh, rows m = 4 (KS i + ks) + c, i = 0..23:  dh_prev[j] = dh z + sum_m dgh[m] W_hh[m, j]
    const float* w_hh = a.w_hh + (SEP ? (long long)(row0 / a.B) * a.agent_stride : 0);      // this pass's agent
    f32x2 wt[48];                                          // (rows m, m+1) pairs
#pragma unroll
    for (int i = 0; i < 24; ++i)
#pragma unroll
        for (int c = 0; c < 2; ++c)
            wt[2 * i + c] = pack2(__ldg(w_hh + (long long)(4 * (KS * i + ks) + 2 * c) * H + j),
                                  __ldg(w_hh + (long long)(4 * (KS * i + ks) + 2 * c + 1) * H + j));
    // cp.async work list: per row CPR chunks of 16 B (H of gates, H / 4 each of h_prev, dh_ext, dh_ext2).  The per-chunk source
    // pointer at t = 0 and its per-step stride are fixed, so they are computed once -- which takes ~35 registers a thread: a
    // 512-thread group, left with 128 registers a thread, recomputes each chunk's source per step instead.
    constexpr bool kChunkList = T < 512;
    constexpr int NCH = (R * CPR + T - 1) / T;
    const float* csrc[NCH]; int cstride[NCH], cdst[NCH], ckind[NCH];
    if constexpr (kChunkList) {
#pragma unroll
        for (int l = 0; l < NCH; ++l) {
            const int c = tid + l * T, rr = c / CPR, ch = c % CPR, row = row_at(rr);
            csrc[l] = nullptr; cstride[l] = 0; cdst[l] = rr * SLOT + ch * 4; ckind[l] = 0;
            if (c < R * CPR && rr < nrows) {
                const long long idx0 = (long long)(row / N) * L * N + (row % N);
                if (ch < H) { csrc[l] = a.gates + idx0 * (4 * H) + ch * 4; cstride[l] = N * 4 * H; }
                else if (ch < H + H / 4) { csrc[l] = a.hidden + (idx0 - N) * H + (ch - H) * 4; cstride[l] = N * H; ckind[l] = 1;
                                           if (a.h0) ckind[l] = 2; }
                else if (ch < H + H / 2) { if (a.dh_ext) { csrc[l] = a.dh_ext + idx0 * H + (ch - H - H / 4) * 4; cstride[l] = N * H; } }
                else { if (a.dh_ext2) { csrc[l] = a.dh_ext2 + idx0 * H + (ch - H - H / 2) * 4; cstride[l] = N * H; } }
            }
        }
    }
    auto issue = [&](int t) {
        if (t >= 0) {
            float* slot = &ring[t % D][0][0];
            if constexpr (kChunkList) {
#pragma unroll
                for (int l = 0; l < NCH; ++l) {
                    if (!csrc[l]) continue;
                    if (ckind[l] != 0 && t == 0) {      // h_prev of the first step: h0 (or zeros, handled by the consumer)
                        if (ckind[l] == 2) cp_async16(slot + cdst[l], a.h0 + (long long)row_at(cdst[l] / SLOT) * H + (cdst[l] % SLOT - 4 * H));
                        continue;
                    }
                    cp_async16(slot + cdst[l], csrc[l] + (long long)t * cstride[l]);
                }
            } else {
                for (int c = tid; c < nrows * CPR; c += T) {
                    const int rr = c / CPR, ch = c % CPR, row = row_at(rr);
                    const long long idx = ((long long)(row / N) * L + t) * N + (row % N);
                    const float* src = nullptr;
                    if (ch < H) src = a.gates + idx * (4 * H) + ch * 4;
                    else if (ch < H + H / 4) {
                        if (t > 0) src = a.hidden + (idx - N) * H + (ch - H) * 4;
                        else if (a.h0) src = a.h0 + (long long)row * H + (ch - H) * 4;     // (zeros without h0: the consumer)
                    } else if (ch < H + H / 2) { if (a.dh_ext) src = a.dh_ext + idx * H + (ch - H - H / 4) * 4; }
                    else if (a.dh_ext2) src = a.dh_ext2 + idx * H + (ch - H - H / 2) * 4;
                    if (src) cp_async16(slot + rr * SLOT + ch * 4, src);
                }
            }
        }
        cp_async_commit();
    };
    for (int idx = tid; idx < 2 * R * G; idx += T) (&sg[0][0][0])[idx] = 0.0f;
    // per-step output pointers of the rows this lane owns, walked backwards one time step (N rows) per iteration
    float* pi_[OWN]; float* ph_[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        pi_[q] = a.dgi + (base[q] + (long long)(L - 1) * N) * G + j;
        ph_[q] = a.dgh + (base[q] + (long long)(L - 1) * N) * G + j;
    }
    const long long ostep = (long long)N * G;
    // early exit (SURVEY 8(f) N3): behind the longest episode of this pass every upstream gradient is masked to zero, so the
    // chain would only produce zeros there -- they are written directly and the chain starts at that episode's last step
    int Lp = L;
    if (a.ep_len) {
        Lp = 1;
        for (int rr = 0; rr < nrows; ++rr) Lp = max(Lp, min(L, __ldg(a.ep_len + row_at(rr) / N)));
        const int tail = L - Lp;
        for (int idx = tid; idx < tail * nrows * (G / 4); idx += T) {
            const int c4 = idx % (G / 4), rr = (idx / (G / 4)) % nrows, t = Lp + idx / ((G / 4) * nrows);
            const int row = row_at(rr);
            const long long off = (((long long)(row / N) * L + t) * N + (row % N)) * G + 4 * c4;
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
                const int rr = ks + KS * q;
                const float* sl = &ring[t % D][rr][0];
                const float g_r = sl[j], g_z = sl[H + j], g_n = sl[2 * H + j], g_hn = sl[3 * H + j];
                const float hprev = (t > 0 || a.h0) ? sl[4 * H + j] : 0.0f;
                float dh = dh_carry[q];
                if (a.dh_ext) dh += sl[5 * H + j];
                if (a.dh_ext2) dh += sl[6 * H + j];
                // h' = (h - n) z + n ; n = tanh(gi_n + r (W_hn h + b_hn)) ; r, z = sigmoid(gi + gh)
                const float dn_pre = dh * (1.0f - g_z) * (1.0f - g_n * g_n);
                const float dz_pre = dh * (hprev - g_n) * g_z * (1.0f - g_z);
                const float dr_pre = dn_pre * g_hn * g_r * (1.0f - g_r);
                const float dghn = dn_pre * g_r;
                dh_dir[q] = dh * g_z;
                float* pi = pi_[q];
                float* ph = ph_[q];
                pi[0] = dr_pre; pi[H] = dz_pre; pi[2 * H] = dn_pre;
                ph[0] = dr_pre; ph[H] = dz_pre; ph[2 * H] = dghn;
                sg[cur][rr][j] = dr_pre; sg[cur][rr][H + j] = dz_pre; sg[cur][rr][2 * H + j] = dghn;
            }
            pi_[q] -= ostep; ph_[q] -= ostep;
        }
        // the refill of the slot of step t+1 (consumed before the previous barrier): early when many rows keep the CTA
        // throughput-bound, behind the FMAs (see the forward kernel) when the chain is latency-bound and the registers allow
        constexpr bool kLateIssue = R <= 2 && T < 512;
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
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&sg[cur][rr][4 * (KS * i + ks)]);
                pab[rr] = ffma2(wt[2 * i], v.x, pab[rr]);
                pcd[rr] = ffma2(wt[2 * i + 1], v.y, pcd[rr]);
            }
        if (kLateIssue) issue(t - (D - 1));
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            float pa, pb, pc, pd;
            unpack2(pab[rr], pa, pb); unpack2(pcd[rr], pc, pd);
            part[rr] = lanes_sum<KS>((pa + pb) + (pc + pd));
        }
#pragma unroll
        for (int q = 0; q < OWN; ++q) dh_carry[q] = dh_dir[q] + lane_pick<KS>(part, q, ks);
        cur ^= 1;
    }
    cp_async_wait<0>();
    if (a.dh0) {
#pragma unroll
        for (int q = 0; q < OWN; ++q)
            if (own[q]) a.dh0[(long long)row_at(ks + KS * q) * H + j] = dh_carry[q];
    }
    __syncthreads();
}

#ifndef MARL_GRU_BWD_CTAS
#define MARL_GRU_BWD_CTAS 2
#endif
constexpr int kGruBwdCtasPerSm = MARL_GRU_BWD_CTAS;      // H = 64: 254 registers x 128 threads and ~55 KB of shared memory: two CTAs fit an SM
// up to two rows per SM: one CTA per row (see marl_agent_unroll_bwd); the same CTA count at every width, so that the row deal
// marl_agent_unroll_fwd plans for it (row_order_bwd) holds
static int gru_bwd_ctas(int rows) { return rows <= kGruBwdCtasPerSm * kNumSMs ? rows : kNumSMs; }
// the largest pass's shared memory (the ring is shallower at 8 rows, so the 4-row pass may need more)
template <int H>
constexpr size_t gru_bwd_smem_max() {
    size_t m = 0;
    for (int R = 1; R <= GruWidth<H>::kMaxRows; R *= 2) m = gru_bwd_smem<H>(R) > m ? gru_bwd_smem<H>(R) : m;
    return m;
}

template <int H, bool SEP>
__global__ void __launch_bounds__(GruWidth<H>::T) gru_unroll_bwd_kernel(GruBwdArgs a) {
    using W = GruWidth<H>;
    pdl_enter();
    extern __shared__ __align__(16) float gru_smem[];
    int begin, count;
    if (SEP) cta_rows_by_agent(a.B, a.N, begin, count);
    else cta_rows(a.B * a.N, 0, begin, count);
    for (int off = 0, n = 0; off < count; off += SEP ? n : W::kMaxRows) {
        n = gru_pass_rows<H, SEP>(begin + off, count - off, a.B);
        if (n == 1) gru_rows_bwd<H, 1, SEP>(a, begin + off, n, gru_smem);
        else if (W::kMaxRows == 2 || n == 2) gru_rows_bwd<H, 2, SEP>(a, begin + off, n, gru_smem);
        else if (W::kMaxRows == 4 || n <= 4) gru_rows_bwd<H, W::rows(4), SEP>(a, begin + off, n, gru_smem);
        else gru_rows_bwd<H, W::rows(8), SEP>(a, begin + off, n, gru_smem);
    }
}

// Forward launch: one CTA per SM and chain group, a thread group per chain.  `smem` (0: what the kernel needs) may ask for more,
// so that the launch has its SMs to itself (gru_fwd_launch_solo); the kernel's opt-in is raised to the largest size asked for.
template <int H>
static void gru_fwd_launch(const GruFwdArgs& ga, int n_ctas, bool sep, cudaStream_t st, size_t smem = 0) {
    using W = GruWidth<H>;
    if (!smem) smem = W::kGroups * gru_fwd_smem<H>(W::kMaxRows);
    static size_t opt_in = 0;
    if (smem > opt_in) {
        cudaFuncSetAttribute(gru_unroll_fwd_kernel<H, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(gru_unroll_fwd_kernel<H, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        opt_in = smem;
    }
    const dim3 grid(n_ctas, (ga.n_chains + W::kGroups - 1) / W::kGroups);
    launch_pdl_prio(kGruPrio, sep ? gru_unroll_fwd_kernel<H, true> : gru_unroll_fwd_kernel<H, false>, grid,
                    dim3(W::T * W::kGroups), smem, st, ga);
}

template <int H>
static void gru_bwd_launch(const GruBwdArgs& ga, int rows, bool sep, cudaStream_t st) {
    constexpr size_t sm = gru_bwd_smem_max<H>();
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(gru_unroll_bwd_kernel<H, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        cudaFuncSetAttribute(gru_unroll_bwd_kernel<H, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        attr_set = true;
    }
    launch_pdl_prio(kGruPrio, sep ? gru_unroll_bwd_kernel<H, true> : gru_unroll_bwd_kernel<H, false>, dim3(gru_bwd_ctas(rows)),
                    dim3(GruWidth<H>::T), sm, st, ga);
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
constexpr int kOrderRows = GruWidth<MARL_H>::kMaxRows;   // rows of a pass level (the H = 64 pass, at every width)
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
    for (int p = 0; p * kOrderRows < mine; ++p) {
        int before = 0, width = 0;                  // rows of level p dealt before this CTA's / in the whole level
        for (int o = lane; o < n_ctas; o += 32) {
            const int w = min(max((int)cnt[o] - kOrderRows * p, 0), kOrderRows);
            width += w;
            if ((p & 1) ? pos[o] > mypos : pos[o] < mypos) before += w;        // the deal runs backwards on odd levels
        }
        before = (int)warp_sum((float)before); width = (int)warp_sum((float)width);
        const int w = min(mine - kOrderRows * p, kOrderRows);
        if (lane < w) {
            const int sorted = level_start + before + lane;
            out[begin + kOrderRows * p + lane] = (int)ep_of_rank[sorted / N] * N + sorted % N;
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

// Fused input layers (csrc/front.cu) of the streams idx[0 .. n) of a shared-network call, as stream k of the launch
static FrontArgs front_args(const marl_dims* d, const marl_unroll_stream* s, const int* idx, int n, int I, int H) {
    FrontArgs fa{};
    fa.rows = d->B * d->L * d->N; fa.I = I; fa.hidden = H;
    for (int k = 0; k < n; ++k) {
        const marl_unroll_stream& u = s[idx[k]];
        fa.s[k].in = agent_input(d, u.obs, u.onehot, u.shift_onehot, u.full_input, input_blocks(0, u.input_flags, u.last_action, u.agent_id));
        fa.s[k].x = u.x; fa.s[k].gi = u.gi;
        fa.s[k].store_x = u.gates != nullptr;
        fa.set[k].w1 = u.params.fc1_w; fa.set[k].b1 = u.params.fc1_b;
        fa.set[k].w_ih = u.params.w_ih; fa.set[k].b_ih = u.params.b_ih;
        fa.set[k].w_ih_t = u.w_ih_t;
    }
    return fa;
}

// ---- split forward -----------------------------------------------------------------------------------------------------------
// A double-Q step (eval on o, target on o_next, eval on o_next continued from the first) at a few hundred agent rows is one
// latency-bound chain: input layers of all three streams -> the 240-step eval chain.  Only the eval/o stream feeds the first 120
// steps, so the forward is split into two levels on disjoint SMs:
//   main lane:    A = input layers of eval/o (~half the SMs, at most two tiles each) -> level 0 = eval/o chain (two rows per CTA)
//                 -> [waits for B] -> level 1 = eval/o_next chain from level 0's h_last
//   forked lane:  B = input layers of the two o_next streams (the other SMs) -> D = target chain (on the SMs B frees)
// A front CTA fills an SM's shared memory, and every recurrence CTA of the split reserves all of it (kernel shared memory size
// below), so no two of these kernels -- nor a GEMM CTA of another stream -- ever share an SM.  Every row is computed by the same
// code on the same inputs as in the one-launch plan: results are bit-identical.
#ifndef MARL_FWD_SPLIT_MAX_ROWS
#define MARL_FWD_SPLIT_MAX_ROWS 170
#endif
// B*N: the SMs a level launch leaves (148 - B*N/2) carry the input layers of the two o_next streams, which must end before level
// 0 does, then the target chain at two rows per thread group (which holds up to 196 rows).  Measured on a B200 at T = 120
// (tools/fwd_split_bench.py, profiles/r10_bench_parent_vs_pr.txt): QMIX step -6.8 % at 160 rows, -0.4 % at 180, +2.5 % at 195
constexpr int kFwdSplitMaxRows = MARL_FWD_SPLIT_MAX_ROWS;
static int g_split_on = -1;
static bool fwd_split_enabled() {
    if (g_split_on < 0) { const char* e = getenv("MARL_B200_FWD_SPLIT"); g_split_on = (e && e[0] == '0') ? 0 : 1; }
    return g_split_on == 1;
}

struct SplitPlan {
    int head, cont, other;       // streams: the continued chain's head (eval/o), its continuation (eval/o_next), the lone chain (target)
    int n_level, n_target;       // recurrence CTAs of each level and of the target chain
    FrontArgs fa, fb;            // input layers of `head` / of `other` and `cont`
};

// The split applies to a shared-network (H = 64) call of exactly three streams, one continuing another, none cut at its episode's
// end, with B*N <= kFwdSplitMaxRows and the fused input-layer kernel available; every other call keeps the one-launch plan.
static bool split_plan(const marl_dims* d, const marl_unroll_stream* s, int n_streams, SplitPlan& p) {
    if (!fwd_split_enabled() || n_streams != 3) return false;
    const int rows = d->B * d->N;
    if (rows > kFwdSplitMaxRows) return false;
    p.cont = -1;
    for (int i = 0; i < n_streams; ++i) {
        const marl_unroll_stream& u = s[i];
        if (u.agent_stride || hidden_width(u.params.hidden) != MARL_H || u.full_input) return false;
        if (u.ep_len || u.padded || u.row_order || u.row_order_bwd) return false;
        if (u.h0_from >= 0) { if (p.cont >= 0) return false; p.cont = i; }
    }
    if (p.cont < 0) return false;
    p.head = s[p.cont].h0_from;
    p.other = 3 - p.head - p.cont;
    if (s[p.head].h0_from >= 0 || !s[p.head].h_last) return false;     // level 1 starts from level 0's h_last
    const InputBlocks b0 = input_blocks(0, s[0].input_flags, s[0].last_action, s[0].agent_id);
    const int I = agent_input_width(d, b0);
    for (int i = 1; i < n_streams; ++i)
        if (agent_input_width(d, input_blocks(0, s[i].input_flags, s[i].last_action, s[i].agent_id)) != I) return false;
    p.n_level = (rows + 1) / 2;
    const int spare = kNumSMs - p.n_level;          // SMs beside a level launch: B's front, then the target chain
    if (spare < 2) return false;
    const int idx_b[2] = {p.other, p.cont};
    p.fb = front_args(d, s, idx_b, 2, I, MARL_H);
    if (!front_plan(p.fb, 2, spare)) return false;
    int grid_b = 0;
    for (int k = 0; k < p.fb.n_sets; ++k) grid_b += p.fb.set[k].n_ctas;
    p.fa = front_args(d, s, &p.head, 1, I, MARL_H);
    if (!front_plan(p.fa, 1, kNumSMs - grid_b)) return false;
    // the target chain: two thread groups per CTA with at most two rows each, on the fewest CTAs that allow it
    const int per = (rows + 2 * spare - 1) / (2 * spare);
    if (per > 2) return false;
    p.n_target = (rows + 2 * per - 1) / (2 * per);
    return true;
}

// The rows of one stream (continued from h0) as `parts` chains, one per thread group of a CTA (two at most): chain c takes the
// episodes [B c / parts, B (c + 1) / parts), addressed through offset pointers, its rows dealt over n_ctas CTAs by water-filling
// on the rows a CTA already carries
static GruFwdArgs single_chain(const marl_dims* d, const marl_unroll_stream& u, const float* h0, int n_ctas, int parts) {
    GruFwdArgs g{};
    g.B = d->B; g.L = d->L; g.N = d->N;
    g.n_chains = parts;
    double load[kNumSMs] = {};
    for (int c = 0; c < parts; ++c) {
        const int b0 = d->B * c / parts, b1 = d->B * (c + 1) / parts;
        const long long step = (long long)b0 * d->L * d->N, row = (long long)b0 * d->N;      // first (b, t, n) / (b, n) of the slice
        g.chain_start[c] = c; g.chain_len[c] = 1;
        g.h0[c] = h0 ? h0 + row * MARL_H : nullptr;
        g.seg[c] = GruSegment{u.gi + step * MARL_G, u.params.w_hh, u.params.b_hh, u.hidden + step * MARL_H,
                              u.gates ? u.gates + step * 4 * MARL_H : nullptr, u.h_last ? u.h_last + row * MARL_H : nullptr, u.ep_len};
        int cnt[kNumSMs] = {};
        water_fill(load, 0, n_ctas, (b1 - b0) * d->N, 1.0, cnt);
        for (int i = 0; i < n_ctas; ++i) { g.rows_of[c][i] = (unsigned short)cnt[i]; load[i] += cnt[i]; }
    }
    g.trace = trace_buffer();
    return g;
}

// A recurrence launch of the split forward: it reserves the whole of the SM's shared memory, so that nothing runs beside it
static void gru_fwd_launch_solo(const GruFwdArgs& ga, int n_ctas, bool pdl, cudaStream_t st) {
    static size_t solo = 0;
    if (!solo) {
        int dev = 0, optin = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaFuncAttributes fa{};
        cudaFuncGetAttributes(&fa, gru_unroll_fwd_kernel<MARL_H, false>);
        solo = (size_t)optin - fa.sharedSizeBytes;
    }
    ProfScope ps_("gru_unroll_fwd_kernel", st);
    const bool keep_ = pdl_small_problem();
    pdl_small_problem() = keep_ && pdl;
    gru_fwd_launch<MARL_H>(ga, n_ctas, false, st, solo);
    pdl_small_problem() = keep_;
}

static int split_forward(const marl_dims* d, const marl_unroll_stream* s, const SplitPlan& p, cudaStream_t st) {
    static cudaEvent_t ev_b[8];
    static int ring = -1;
    if (ring < 0) { for (auto& e : ev_b) cudaEventCreateWithFlags(&e, cudaEventDisableTiming); ring = 0; }
    ring = (ring + 1) & 7;
    ForkJoin fj(st, 2);
    cudaStream_t side = fj.lane(1);
    int rc = front_launch(p.fa, 1, kGruPrio, st);                  // A
    if (rc) return rc;
    if ((rc = front_launch(p.fb, 2, kGruPrio, side))) return rc;    // B
    cudaEventRecord(ev_b[ring], side);
    // level 0 behind A (programmatic: its CTAs take A's SMs as A's CTAs leave)
    gru_fwd_launch_solo(single_chain(d, s[p.head], s[p.head].h0, p.n_level, 1), p.n_level, true, st);
    MARL_LAUNCH_CHECK();
    // the target chain behind B, on the SMs B frees: its rows in two slices, one per thread group, at most two rows per group
    // (a single group with three rows, the four-row pass, takes twice as long per step as one with two)
    gru_fwd_launch_solo(single_chain(d, s[p.other], s[p.other].h0, p.n_target, 2), p.n_target, true, side);
    MARL_LAUNCH_CHECK();
    // level 1 from level 0's final hidden state.  A plain launch: launched programmatically its CTAs would become resident beside
    // level 0 as soon as B ends and take the SMs the target chain is about to use
    cudaStreamWaitEvent(st, ev_b[ring], 0);
    gru_fwd_launch_solo(single_chain(d, s[p.cont], s[p.head].h_last, p.n_level, 1), p.n_level, false, st);
    MARL_LAUNCH_CHECK();
    fj.join();
    return MARL_OK;
}

}  // namespace marl

using namespace marl;

// A/B switch of the split forward (MARL_B200_FWD_SPLIT, default on); returns the previous setting
extern "C" int marl_fwd_split_enable(int on) {
    const int prev = fwd_split_enabled() ? 1 : 0;
    g_split_on = on ? 1 : 0;
    return prev;
}

// 1 when marl_agent_unroll_fwd would run these streams as the split forward (five launches for the input layers and the
// recurrence instead of two), 0 otherwise
extern "C" int marl_agent_unroll_fwd_split(const marl_dims* d, const marl_unroll_stream* s, int n_streams) {
    if (check_dims(d) || !s || n_streams < 1 || n_streams > kMaxStreams) return MARL_EINVAL;
    SplitPlan p;
    return split_plan(d, s, n_streams, p) ? 1 : 0;
}

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
    // rnn_hidden_dim: one width for every stream of the call
    const int H = hidden_width(s[0].params.hidden), G = 3 * H;
    if (H < 0) return MARL_EINVAL;
    for (int i = 0; i < n_streams; ++i)
        if (hidden_width(s[i].params.hidden) != H) return MARL_EINVAL;
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
                const int nb = gru_bwd_ctas(rows);      // (the same CTA count at every width)
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
        LinearFwd f = agent_layer(d, in, s[i].params.fc1_w, I, s[i].params.fc1_b, s[i].x, H, stride);
        f.relu = 1;
        return f;
    };
    auto ih_of = [&](int i) {
        const LinOperand in = sep ? plain_operand(s[i].x, d->N * H, H, H) : plain_operand(s[i].x, H, H);
        return agent_layer(d, in, s[i].params.w_ih, H, s[i].params.b_ih, s[i].gi, G, stride);
    };
    bool grouped = false;
    SplitPlan split;
    const bool split_on = split_plan(d, s, n_streams, split);
    if (split_on) {
        const int rc = split_forward(d, s, split, st);
        if (rc) return rc;
        grouped = true;
    } else if (!sep) {      // (the fused input-layer kernel stages one shared weight set: separated streams take the unfused path)
        // fused path (csrc/front.cu): both layers of every stream in ONE persistent launch, x handed from the first GEMM to the
        // second through tensor memory
        const int idx[kMaxStreams] = {0, 1, 2, 3};
        FrontArgs fa = front_args(d, s, idx, n_streams, I, H);
        if (front_plan(fa, n_streams)) {
            const int rc = front_launch(fa, n_streams, kGruPrio, st);
            if (rc) return rc;
            grouped = true;
        }
    }
    if (!grouped) {
        for (int i = 0; i < n_streams; ++i)
            if (s[i].w_ih_t) {
                const int rc = transpose_weights(s[i].params.w_ih, H, 0, G, H, s[i].w_ih_t, st);
                if (rc) return rc;
            }
    }
    if (!grouped && !sep && H == MARL_H && tgemm_enabled()) {
        // TMA path: the streams of one layer are ONE grouped launch of persistent CTAs (csrc/tgemm.cu): 2 launches
        // instead of 2 x n_streams on forked streams.  (Other widths take the register-staged kernels of linear.cu: the
        // TMA builders have only been checked on the 64-wide agent layers.)
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
    if (!split_on) {
        // one CTA per SM; each CTA advances its share of every chain side by side (one 128-thread group per chain)
        ProfScope ps_("gru_unroll_fwd_kernel", st);
        ga.trace = trace_buffer();
        if (order_lane) order_lane->join();
        switch (H) {
        case 32: gru_fwd_launch<32>(ga, n_ctas, sep, st); break;
        case 64: gru_fwd_launch<64>(ga, n_ctas, sep, st); break;
        default: gru_fwd_launch<128>(ga, n_ctas, sep, st); break;
        }
    }
    MARL_LAUNCH_CHECK();
    // phase C.  (The fork / join pair stays even when a fused mixer evaluates the heads and nothing is launched here: it takes the
    // programmatic launch edge between the recurrence and the mixing kernel, whose 480 early-resident CTAs otherwise sit on the
    // SMs beside the last steps of the recurrence -- measured 333 us per step with the pair, 345-354 us without.)
    ForkJoin fc(st, n_streams);
    for (int i = 0; i < n_streams; ++i) {
        if (!s[i].q) continue;
        cudaStream_t st = fc.lane(i);
        const LinOperand in = sep ? plain_operand(s[i].hidden, d->N * H, H, H) : plain_operand(s[i].hidden, H, H);
        int rc = linear_fwd(agent_layer(d, in, s[i].params.fc2_w, H, s[i].params.fc2_b, s[i].q, d->A, stride), st);
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
    const int H = hidden_width(a->params.hidden), G = 3 * H;
    if (H < 0) return MARL_EINVAL;
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
        g.dy = a->dq; g.lddy = rp * d->A; g.dy_bs = zs(d->A); g.w = a->params.fc2_w; g.ldw = H; g.w_bs = stride; g.w_col0 = 0;
        g.dx = a->dhext; g.lddx = rp * H; g.dx_bs = zs(H); g.M = M; g.N = d->A; g.K = H; g.batch = nb;
        if ((rc = linear_dgrad(g, st))) return rc;
    }
    GruBwdArgs ga{a->gates, a->hidden, a->dq ? a->dhext : nullptr, a->dhidden, a->params.w_hh, a->h0, a->dgi, a->dgh, a->dh0,
                  d->B, d->L, d->N, a->ep_len, (a->ep_len && d->B <= kMaxOrderEpisodes) ? a->row_order : nullptr, stride};
    const int rows = d->B * d->N;
    {
        ProfScope ps_("gru_unroll_bwd_kernel", st);
        const bool keep_ = pdl_small_problem();
        // measured: launched programmatically the 148 recurrence CTAs come up while the producer still runs and the
        // step gets 10-27 us slower on every config; a plain launch here, PDL for its consumers
        pdl_small_problem() = false;
        // up to two rows per SM: one CTA per row -- two co-resident one-row CTAs overlap each other's latency, where one CTA with two
        // rows serialises 2 x 96 packed FMAs per thread on the dependent chain (the 12 two-row CTAs of config 2 ended the kernel)
        switch (H) {
        case 32: gru_bwd_launch<32>(ga, rows, sep, st); break;
        case 64: gru_bwd_launch<64>(ga, rows, sep, st); break;
        default: gru_bwd_launch<128>(ga, rows, sep, st); break;
        }
        pdl_small_problem() = keep_;
    }
    MARL_LAUNCH_CHECK();
    LinearWgrad w_fc2{}, w_hh{}, w_ih{}, w_fc1{}, w_h0{};
    LinearDgrad g_dx{};
    // dW2 += dq^T h ; db2 += colsum(dq)
    w_fc2.dy = a->dq; w_fc2.lddy = rp * d->A; w_fc2.dy_bs = zs(d->A); w_fc2.in = plain_operand(a->hidden, rp * H, H, zs(H));
    w_fc2.dw = a->grads.fc2_w; w_fc2.ldw = H; w_fc2.db = a->grads.fc2_b; w_fc2.M = M; w_fc2.N = d->A; w_fc2.batch = nb;
    w_fc2.dw_bs = stride; w_fc2.db_bs = stride;
    // dW_hh += dgh^T . h_{t-1} (hidden shifted by one step, zeros at t = 0) ; db_hh
    w_hh.dy = a->dgh; w_hh.lddy = rp * G; w_hh.dy_bs = zs(G);
    {
        LinOperand in{};
        in.x = nullptr; in.K1 = 0; in.x2 = a->hidden; in.ldx2 = rp * H; in.K2 = H; in.x2_bs = zs(H);
        in.x2_shift = sep ? 1 : d->N; in.x2_period = sep ? d->L : d->L * d->N; in.onehot_mod = 0;
        w_hh.in = in;
    }
    w_hh.dw = a->grads.w_hh; w_hh.ldw = H; w_hh.db = a->grads.b_hh; w_hh.M = M; w_hh.N = G; w_hh.batch = nb;
    w_hh.dw_bs = stride; w_hh.db_bs = stride;
    // the t = 0 rows see h0 instead of zeros: one [N x H] problem per episode (separated: one [B x H] problem per agent)
    w_h0.dw = a->grads.w_hh; w_h0.ldw = H; w_h0.db = nullptr; w_h0.N = G;
    if (sep) {
        w_h0.dy = a->dgh; w_h0.lddy = d->L * d->N * G; w_h0.dy_bs = G;
        w_h0.in = plain_operand(a->h0, d->N * H, H, H);
        w_h0.M = d->B; w_h0.batch = d->N; w_h0.dw_bs = stride;
    } else {
        w_h0.dy = a->dgh; w_h0.lddy = G; w_h0.dy_bs = (long long)d->L * d->N * G;
        w_h0.in = plain_operand(a->h0, H, H, (long long)d->N * H);
        w_h0.M = d->N; w_h0.batch = d->B;
    }
    // dW_ih += dgi^T . x ; db_ih
    w_ih.dy = a->dgi; w_ih.lddy = rp * G; w_ih.dy_bs = zs(G); w_ih.in = plain_operand(a->x, rp * H, H, zs(H));
    w_ih.dw = a->grads.w_ih; w_ih.ldw = H; w_ih.db = a->grads.b_ih; w_ih.M = M; w_ih.N = G; w_ih.batch = nb;
    w_ih.dw_bs = stride; w_ih.db_bs = stride;
    // dx = (dgi . W_ih) * (x > 0)
    g_dx.dy = a->dgi; g_dx.lddy = rp * G; g_dx.dy_bs = zs(G); g_dx.w = a->params.w_ih; g_dx.ldw = H; g_dx.w_bs = stride;
    g_dx.w_col0 = 0;
    g_dx.dx = a->dx; g_dx.lddx = rp * H; g_dx.dx_bs = zs(H); g_dx.relu_src = a->x; g_dx.ldrs = rp * H; g_dx.rs_bs = zs(H);
    g_dx.M = M; g_dx.N = G; g_dx.K = H; g_dx.batch = nb;
    g_dx.wt = a->w_ih_t; g_dx.ldwt = G;      // W_ih transposed by this step's forward pass (both operands then stage with 128-bit stores)
    // dW1 += dx^T . [obs | last_action | agent_id] ; db1
    w_fc1.dy = a->dx; w_fc1.lddy = rp * H; w_fc1.dy_bs = zs(H);
    w_fc1.in = sep ? separated_input(d, a->obs, a->onehot, a->shift_onehot, a->last_action, a->agent_id)
                   : agent_input(d, a->obs, a->onehot, a->shift_onehot, a->full_input, blk);
    w_fc1.dw = a->grads.fc1_w; w_fc1.ldw = I; w_fc1.db = a->grads.fc1_b; w_fc1.M = M; w_fc1.N = H; w_fc1.batch = nb;
    w_fc1.dw_bs = stride; w_fc1.db_bs = stride;

    if (!sep && H == MARL_H && tgemm_enabled()) {
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
