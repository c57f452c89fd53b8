// Batched acting (controller/share_params.py:37-72 for every (env, agent) row in one launch, with the shared network
// or, as SeparatedMAC does at :419-453, with each agent's own network) and the per-step
// bookkeeping of the batched multi-step rollout (rollout.py:52-149 for all instances at once).
#include <math.h>

#include "common.cuh"
#include "../../include/marl_b200.h"
#include "philox.cuh"
#include "profile.h"

namespace marl {

constexpr int kActThreads = 256;
constexpr int kActRows = 32;       // rows per tile: thread (jg, rg) owns rows {rg, rg + 16} x columns {jg + 16 c}
constexpr int kActKC = 32;         // input columns staged per chunk
constexpr int kHP = MARL_H + 1;    // odd row stride of the 64-wide operands: 16 column groups read 16 distinct banks

// Shared-memory carve-up (in floats).  Every weight stays in its global [out, in] layout; rows are padded to an odd stride.
struct ActLayout {
    int I, Ip, A, qw;
    int w1, b1, wih, whh, bih, bhh, w2, b2, in, xq, h, total;
};

inline ActLayout act_layout(int I, int A) {
    ActLayout l;
    l.I = I; l.Ip = I | 1; l.A = A; l.qw = A > kHP ? A : kHP;
    int o = 0;
    l.w1 = o;  o += MARL_H * l.Ip;
    l.b1 = o;  o += MARL_H;
    l.wih = o; o += MARL_G * kHP;
    l.whh = o; o += MARL_G * kHP;
    l.bih = o; o += MARL_G;
    l.bhh = o; o += MARL_G;
    l.w2 = o;  o += A * kHP;
    l.b2 = o;  o += A;
    l.in = o;  o += kActRows * (kActKC + 1);
    l.xq = o;  o += kActRows * l.qw;      // relu(fc1) tile, then the q tile
    l.h = o;   o += kActRows * kHP;
    l.total = o;
    return l;
}

struct ActArgs {
    int rows, n_envs, N, A, O;
    int last_action, agent_id;                              // input blocks present (marl_agent_act: both)
    const float* obs; const float* last; const float* avail;
    const float* h_in; float* h_out;                       // may alias
    const unsigned char* explore; const long long* random_action;
    const double* explore_u; const double* choice_u; double eps;
    const int* gate;
    long long* action; float* onehot; float* q;
};

// Philox exploration form (marl_act_philox): the selection thread of row e*N + n draws its own pair.
struct ActPhilox {
    unsigned long long seed, episode_base;
    int step;
    const double* eps_table; int eps_len;
};

// The uniform form's random action: the min(floor(u * cnt), cnt - 1)-th of the cnt available actions, 0 when cnt == 0.
// The Philox form calls it; the uniform form keeps its own copy inline in agent_act_kernel, so that its code is what it
// was before the Philox form existed.
__device__ __forceinline__ int kth_available(const float* av, int A, int cnt, double u) {
    int best = 0;
    if (cnt > 0) {
        const double c = (double)cnt;
        const int kth = (int)fmin(floor(u * c), c - 1.0);
        for (int k = 0, seen = 0; k < A; ++k)
            if (!av || av[k] != 0.0f) {
                if (seen == kth) { best = k; break; }
                ++seen;
            }
    }
    return best;
}

constexpr int kActMaxAgents = 128;  // parameter sets one separated launch carries (8 KB of kernel parameters)

template <int kSets>
struct ActParams { marl_agent_params p[kSets]; };

// kSets == 1: the shared agent; a tile is 32 consecutive rows, tiles dealt round-robin.
// kSets > 1: agent n's own weights; a tile is up to 32 instances of ONE agent (rows e*N + n), tiles are agent-major and
// every CTA takes a contiguous range of them, so it restages weights only when its agent changes.
// kPhilox: exploration from ph (a's four exploration pointers are NULL); otherwise ph is not read.
template <int kSets, bool kPhilox>
__global__ void __launch_bounds__(kActThreads) agent_act_kernel(const __grid_constant__ ActParams<kSets> ps, ActArgs a,
                                                                ActLayout l, ActPhilox ph) {
    constexpr bool kSep = kSets > 1;
    if (a.gate && *(volatile const int*)a.gate == 0) return;
    extern __shared__ float sm[];
    __shared__ int act_s[kActRows];
    float *w1 = sm + l.w1, *b1 = sm + l.b1, *wih = sm + l.wih, *whh = sm + l.whh, *bih = sm + l.bih, *bhh = sm + l.bhh;
    float *w2 = sm + l.w2, *b2 = sm + l.b2, *ins = sm + l.in, *xq = sm + l.xq, *hs = sm + l.h;
    const int tid = threadIdx.x, A = a.A, O = a.O, I = l.I, Ip = l.Ip;

    auto stage = [&](const marl_agent_params& p) {
        for (int i = tid; i < MARL_H * I; i += kActThreads) { const int j = i / I; w1[j * Ip + (i - j * I)] = __ldg(p.fc1_w + i); }
        for (int i = tid; i < MARL_G * MARL_H; i += kActThreads) {
            const int g = i >> 6, k = i & 63;
            wih[g * kHP + k] = __ldg(p.w_ih + i);
            whh[g * kHP + k] = __ldg(p.w_hh + i);
        }
        for (int i = tid; i < A * MARL_H; i += kActThreads) w2[(i >> 6) * kHP + (i & 63)] = __ldg(p.fc2_w + i);
        for (int i = tid; i < MARL_H; i += kActThreads) b1[i] = __ldg(p.fc1_b + i);
        for (int i = tid; i < MARL_G; i += kActThreads) { bih[i] = __ldg(p.b_ih + i); bhh[i] = __ldg(p.b_hh + i); }
        for (int i = tid; i < A; i += kActThreads) b2[i] = __ldg(p.fc2_b + i);
    };

    const int jg = tid & 15, rg = tid >> 4;
    const int K = O + (a.last_action ? A : 0);   // [obs | last action]; the agent-id block is one column, added below
    const int per_agent = (a.n_envs + kActRows - 1) / kActRows;
    const int ntiles = kSep ? per_agent * a.N : (a.rows + kActRows - 1) / kActRows;
    const int t_begin = kSep ? (int)((long long)ntiles * blockIdx.x / gridDim.x) : blockIdx.x;
    const int t_end = kSep ? (int)((long long)ntiles * (blockIdx.x + 1) / gridDim.x) : ntiles;
    const int t_step = kSep ? 1 : gridDim.x;
    int staged = -1;
    if (!kSep) stage(ps.p[0]);
    for (int tile = t_begin; tile < t_end; tile += t_step) {
        // tile row r is global row base + r * stride, r < cnt; the tile's agent is n_tile (separated) or row % N
        int n_tile = 0, stride = 1, cnt;
        long long base;
        if (kSep) {
            n_tile = tile / per_agent;
            const int e0 = (tile - n_tile * per_agent) * kActRows;
            base = (long long)e0 * a.N + n_tile; stride = a.N; cnt = min(kActRows, a.n_envs - e0);
            if (n_tile != staged) {
                __syncthreads();          // the previous agent's weights are no longer read
                stage(ps.p[n_tile]);
                staged = n_tile;
            }
        } else {
            base = (long long)tile * kActRows; cnt = min(kActRows, a.rows - (int)base);
        }
        __syncthreads();                  // weights staged / the previous tile's q tile consumed
        for (int i = tid; i < kActRows * MARL_H; i += kActThreads) {
            const int r = i >> 6, k = i & 63;
            hs[r * kHP + k] = r < cnt ? a.h_in[(base + (long long)r * stride) * MARL_H + k] : 0.f;
        }
        // ---- x = relu(fc1 [obs | last | eye(N)[n]] + b1)
        float acc[2][4];
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[0][c] = acc[1][c] = b1[jg + 16 * c];
        for (int k0 = 0; k0 < K; k0 += kActKC) {
            const int kc = min(kActKC, K - k0);
            __syncthreads();
            for (int i = tid; i < kActRows * kActKC; i += kActThreads) {
                const int r = i / kActKC, kk = i % kActKC, k = k0 + kk;
                const long long row = base + (long long)r * stride;
                float v = 0.f;
                if (r < cnt && kk < kc)
                    v = k < O ? __ldg(a.obs + row * O + k) : __ldg(a.last + row * A + (k - O));
                ins[r * (kActKC + 1) + kk] = v;
            }
            __syncthreads();
            for (int kk = 0; kk < kc; ++kk) {
                const float v0 = ins[rg * (kActKC + 1) + kk], v1 = ins[(rg + 16) * (kActKC + 1) + kk];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float w = w1[(jg + 16 * c) * Ip + k0 + kk];
                    acc[0][c] = fmaf(w, v0, acc[0][c]);
                    acc[1][c] = fmaf(w, v1, acc[1][c]);
                }
            }
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = rg + 16 * rr, n = kSep ? n_tile : ((int)base + r) % a.N;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = jg + 16 * c;
                xq[r * kHP + j] = fmaxf(a.agent_id ? acc[rr][c] + w1[j * Ip + K + n] : acc[rr][c], 0.f);
            }
        }
        __syncthreads();
        // ---- GRUCell, gate order r, z, n (torch)
        float gi[2][3][4], gh[2][3][4];
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                gi[0][g][c] = gi[1][g][c] = bih[g * MARL_H + jg + 16 * c];
                gh[0][g][c] = gh[1][g][c] = bhh[g * MARL_H + jg + 16 * c];
            }
#pragma unroll 4
        for (int k = 0; k < MARL_H; ++k) {
            const float x0 = xq[rg * kHP + k], x1 = xq[(rg + 16) * kHP + k];
            const float h0 = hs[rg * kHP + k], h1 = hs[(rg + 16) * kHP + k];
#pragma unroll
            for (int g = 0; g < 3; ++g)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int o = (g * MARL_H + jg + 16 * c) * kHP + k;
                    const float wi = wih[o], wh = whh[o];
                    gi[0][g][c] = fmaf(wi, x0, gi[0][g][c]); gi[1][g][c] = fmaf(wi, x1, gi[1][g][c]);
                    gh[0][g][c] = fmaf(wh, h0, gh[0][g][c]); gh[1][g][c] = fmaf(wh, h1, gh[1][g][c]);
                }
        }
        float hn[2][4];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float r = sigmoidf_acc(gi[rr][0][c] + gh[rr][0][c]);
                const float z = sigmoidf_acc(gi[rr][1][c] + gh[rr][1][c]);
                const float nn = tanhf(gi[rr][2][c] + r * gh[rr][2][c]);
                hn[rr][c] = (1.f - z) * nn + z * hs[(rg + 16 * rr) * kHP + jg + 16 * c];
            }
        __syncthreads();                  // every read of x and h done
#pragma unroll
        for (int rr = 0; rr < 2; ++rr)
#pragma unroll
            for (int c = 0; c < 4; ++c) hs[(rg + 16 * rr) * kHP + jg + 16 * c] = hn[rr][c];
        __syncthreads();
        for (int i = tid; i < kActRows * MARL_H; i += kActThreads) {
            const int r = i >> 6, k = i & 63;
            if (r < cnt) a.h_out[(base + (long long)r * stride) * MARL_H + k] = hs[r * kHP + k];
        }
        // ---- q = fc2 h' + b2 (the q tile reuses the x tile)
        for (int i = tid; i < kActRows * A; i += kActThreads) {
            const int r = i / A, act = i - r * A;
            float s = b2[act];
#pragma unroll 8
            for (int k = 0; k < MARL_H; ++k) s = fmaf(w2[act * kHP + k], hs[r * kHP + k], s);
            xq[r * A + act] = s;
            if (a.q && r < cnt) a.q[(base + (long long)r * stride) * A + act] = s;
        }
        __syncthreads();
        // ---- masked first maximum, then the exploration forms
        if (tid < cnt) {
            const long long row = base + (long long)tid * stride;
            const float* av = a.avail ? a.avail + row * A : nullptr;
            int best = 0, cnt_av = 0;
            float bv = -INFINITY;
            for (int k = 0; k < A; ++k) {
                const bool ok = !av || av[k] != 0.0f;
                const float v = ok ? xq[tid * A + k] : -INFINITY;
                if (v > bv) { bv = v; best = k; }          // strict: first maximum; all masked -> 0 like th.argmax
                cnt_av += ok;
            }
            if constexpr (kPhilox) {
                const int e = (int)(row / a.N), n = (int)(row - (long long)e * a.N);
                const double eps = ph.eps_table ? ph.eps_table[min(e, ph.eps_len - 1)] : a.eps;
                double eu, cu;
                philox_act_uniforms(ph.seed, ph.episode_base + (unsigned long long)e, ph.step, n, eu, cu);
                if (eu < eps) best = kth_available(av, A, cnt_av, cu);
            } else if (a.explore) {
                if (a.explore[row]) best = (int)a.random_action[row];
            } else if (a.explore_u && a.explore_u[row] < a.eps) {
                best = 0;                                   // no available action: action 0
                if (cnt_av > 0) {
                    const double c = (double)cnt_av;
                    const int kth = (int)fmin(floor(a.choice_u[row] * c), c - 1.0);
                    for (int k = 0, seen = 0; k < A; ++k)
                        if (!av || av[k] != 0.0f) {
                            if (seen == kth) { best = k; break; }
                            ++seen;
                        }
                }
            }
            act_s[tid] = best;
            a.action[row] = best;
        }
        if (a.onehot) {
            __syncthreads();
            for (int i = tid; i < kActRows * A; i += kActThreads) {
                const int r = i / A, act = i - r * A;
                if (r < cnt) a.onehot[(base + (long long)r * stride) * A + act] = act == act_s[r] ? 1.0f : 0.0f;
            }
        }
    }
}

// One warp per instance.  Phase t (1 <= t <= T) closes step t-1 for the instances that acted in it (what env.step
// returned, the one-hot of their action, and the observation / state / availability read after it) and opens step t
// for the instances still active (the getters' values are the step's o / s / avail_u).
constexpr int kRecWarps = 8;

struct RecArgs {
    marl_dims d; int t; marl_episode_f32 ep;
    const float* obs; const float* state; const float* avail;
    const long long* action; const float* onehot; const double* reward; const unsigned char* terminated;
    unsigned char* active; float* last; double* reward_sum; int* counters; int* active_host;
};

__device__ __forceinline__ void warp_copy(float* dst, const float* src, int n, int lane) {
    for (int i = lane; i < n; i += 32) dst[i] = src[i];
}

__global__ void __launch_bounds__(kRecWarps * 32) rollout_record_kernel(RecArgs a) {
    const int lane = threadIdx.x & 31, e = blockIdx.x * kRecWarps + (threadIdx.x >> 5);
    const int N = a.d.N, A = a.d.A, O = a.d.O, S = a.d.S, T = a.d.L, t = a.t;
    bool now = false;
    if (e < a.d.B) {
        const bool was = a.active[e] != 0;
        now = was;
        if (t > 0 && was) {
            const int s = t - 1;
            const long long eo = (long long)e * T + s;      // (instance, step) record index
            const bool term = a.terminated[e] != 0;
            now = !term;
            for (int i = lane; i < N; i += 32) a.ep.u[eo * N + i] = a.action[(long long)e * N + i];
            warp_copy(a.ep.u_onehot + eo * N * A, a.onehot + (long long)e * N * A, N * A, lane);
            warp_copy(a.last + (long long)e * N * A, a.onehot + (long long)e * N * A, N * A, lane);
            warp_copy(a.ep.o_next + eo * N * O, a.obs + (long long)e * N * O, N * O, lane);
            warp_copy(a.ep.s_next + eo * S, a.state + (long long)e * S, S, lane);
            warp_copy(a.ep.avail_u_next + eo * N * A, a.avail + (long long)e * N * A, N * A, lane);
            if (lane == 0) {
                const double r = a.reward[e];
                a.ep.r[eo] = (float)r;
                a.ep.terminated[eo] = term ? 1.0f : 0.0f;
                a.ep.padded[eo] = 0.0f;
                a.reward_sum[e] += r;
                a.active[e] = now ? 1 : 0;
            }
        }
        if (t < T && now) {
            const long long eo = (long long)e * T + t;
            warp_copy(a.ep.o + eo * N * O, a.obs + (long long)e * N * O, N * O, lane);
            warp_copy(a.ep.s + eo * S, a.state + (long long)e * S, S, lane);
            warp_copy(a.ep.avail_u + eo * N * A, a.avail + (long long)e * N * A, N * A, lane);
        }
    }
    if (t >= T) return;
    // instances active at the start of step t: counters[t], and their running sum counters[T] (the environment steps)
    const int here = __syncthreads_count(lane == 0 && now);
    if (threadIdx.x == 0) {
        if (here) { atomicAdd(a.counters + t, here); atomicAdd(a.counters + T, here); }
        if (a.active_host) {                                // the last CTA publishes the step's count to the host word
            __threadfence();
            const unsigned ticket = atomicAdd((unsigned*)(a.counters + T + 1), 1u);
            if (ticket == gridDim.x - 1) {
                __threadfence();
                *(volatile int*)a.active_host = atomicAdd(a.counters + t, 0);
                __threadfence_system();
                a.counters[T + 1] = 0;
            }
        }
    }
}

}  // namespace marl

using namespace marl;

// Validates the on-chip footprint of one parameter set of input width I and launches agent_act_kernel<kSets, kPhilox>.
template <int kSets, bool kPhilox>
static int act_launch(const char* name, const ActParams<kSets>& ps, const ActArgs& a, const ActPhilox& ph, int I,
                      long long tiles, void* stream) {
    const ActLayout l = act_layout(I, a.A);
    const size_t smem = (size_t)l.total * sizeof(float);
    int dev = 0, sms = 0, optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return (int)e;
    if (smem + kActRows * sizeof(int) > (size_t)optin) return MARL_EINVAL;      // weights of this shape do not fit on chip
    if (tiles == 0) return MARL_OK;
    static size_t smem_set[64] = {};
    static int blocks_per_sm[64] = {};
    static size_t blocks_for[64] = {};
    const int slot = dev & 63;
    auto kernel = agent_act_kernel<kSets, kPhilox>;
    if (smem_set[slot] < smem) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        smem_set[slot] = smem;
    }
    if (blocks_for[slot] != smem) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm[slot], kernel, kActThreads, smem);
        if (e != cudaSuccess) return (int)e;
        blocks_for[slot] = smem;
    }
    const long long cap = (long long)sms * (blocks_per_sm[slot] > 0 ? blocks_per_sm[slot] : 1);
    { ProfScope ps_(name, (cudaStream_t)stream);
      kernel<<<(int)(tiles < cap ? tiles : cap), kActThreads, smem, (cudaStream_t)stream>>>(ps, a, l, ph); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

static bool params_complete(const marl_agent_params& p) {
    return p.fc1_w && p.fc1_b && p.w_ih && p.w_hh && p.b_ih && p.b_hh && p.fc2_w && p.fc2_b;
}

// The checks every marl_agent_act* call makes, then the launch: the shared agent (kSep false, p -> one parameter set)
// or one network per agent (p -> N sets).
template <bool kSep, bool kPhilox>
static int act_call(int n_envs, int N, int A, int O, int last_action, int agent_id, const marl_agent_params* p,
                    const float* obs, const float* last_onehot, const float* avail, const float* h_in, float* h_out,
                    const unsigned char* explore, const long long* random_action, const double* explore_u,
                    const double* choice_u, double eps, const int* gate, long long* action, float* onehot, float* q,
                    const ActPhilox& ph, void* stream) {
    if (n_envs < 0 || N <= 0 || (kSep && N > kActMaxAgents) || A <= 0 || O < 0 || !p || !obs || !h_in || !h_out || !action)
        return MARL_EINVAL;
    if (last_action && !last_onehot) return MARL_EINVAL;
    for (int n = 0; n < (kSep ? N : 1); ++n)
        if (!params_complete(p[n])) return MARL_EINVAL;
    if (!explore != !random_action || !explore_u != !choice_u || (explore && explore_u)) return MARL_EINVAL;
    const long long rows = (long long)n_envs * N;
    if (rows > 0x7fffffffLL) return MARL_EINVAL;
    const ActArgs a{(int)rows, n_envs, N, A, O, last_action ? 1 : 0, agent_id ? 1 : 0, obs, last_onehot, avail, h_in, h_out,
                    explore, random_action, explore_u, choice_u, eps, gate, action, onehot, q};
    const int I = O + (last_action ? A : 0) + (agent_id ? N : 0);
    if constexpr (kSep) {
        ActParams<kActMaxAgents> ps{};
        for (int n = 0; n < N; ++n) ps.p[n] = p[n];
        return act_launch<kActMaxAgents, kPhilox>("agent_act_separated_kernel", ps, a, ph, I,
                                                  (long long)N * ((n_envs + kActRows - 1) / kActRows), stream);
    } else {
        const ActParams<1> ps{{*p}};
        return act_launch<1, kPhilox>("agent_act_kernel", ps, a, ph, I, (rows + kActRows - 1) / kActRows, stream);
    }
}

static bool philox_ok(const marl_act_philox* d, ActPhilox& ph) {
    if (!d || d->step < 0 || (d->eps_table && d->eps_len < 1)) return false;
    ph = ActPhilox{d->seed, d->episode_base, d->step, d->eps_table, d->eps_len};
    return true;
}

extern "C" int marl_agent_act_input(int n_envs, int N, int A, int O, int last_action, int agent_id,
                                    const marl_agent_params* p, const float* obs, const float* last_onehot,
                                    const float* avail, const float* h_in, float* h_out, const unsigned char* explore,
                                    const long long* random_action, const double* explore_u, const double* choice_u,
                                    double eps, const int* gate, long long* action, float* onehot, float* q, void* stream) {
    return act_call<false, false>(n_envs, N, A, O, last_action, agent_id, p, obs, last_onehot, avail, h_in, h_out, explore,
                                  random_action, explore_u, choice_u, eps, gate, action, onehot, q, ActPhilox{}, stream);
}

extern "C" int marl_agent_act(int n_envs, int N, int A, int O, const marl_agent_params* p, const float* obs,
                              const float* last_onehot, const float* avail, const float* h_in, float* h_out,
                              const unsigned char* explore, const long long* random_action, const double* explore_u,
                              const double* choice_u, double eps, const int* gate, long long* action, float* onehot,
                              float* q, void* stream) {
    return marl_agent_act_input(n_envs, N, A, O, 1, 1, p, obs, last_onehot, avail, h_in, h_out, explore, random_action,
                                explore_u, choice_u, eps, gate, action, onehot, q, stream);
}

extern "C" int marl_agent_act_separated(int n_envs, int N, int A, int O, int last_action, int agent_id,
                                        const marl_agent_params* p, const float* obs, const float* last_onehot,
                                        const float* avail, const float* h_in, float* h_out, const unsigned char* explore,
                                        const long long* random_action, const double* explore_u, const double* choice_u,
                                        double eps, const int* gate, long long* action, float* onehot, float* q,
                                        void* stream) {
    return act_call<true, false>(n_envs, N, A, O, last_action, agent_id, p, obs, last_onehot, avail, h_in, h_out, explore,
                                 random_action, explore_u, choice_u, eps, gate, action, onehot, q, ActPhilox{}, stream);
}

extern "C" int marl_agent_act_philox(int n_envs, int N, int A, int O, int last_action, int agent_id,
                                     const marl_agent_params* p, const float* obs, const float* last_onehot,
                                     const float* avail, const float* h_in, float* h_out, const marl_act_philox* philox,
                                     double eps, const int* gate, long long* action, float* onehot, float* q,
                                     void* stream) {
    ActPhilox ph;
    if (!philox_ok(philox, ph)) return MARL_EINVAL;
    return act_call<false, true>(n_envs, N, A, O, last_action, agent_id, p, obs, last_onehot, avail, h_in, h_out, nullptr,
                                 nullptr, nullptr, nullptr, eps, gate, action, onehot, q, ph, stream);
}

extern "C" int marl_agent_act_separated_philox(int n_envs, int N, int A, int O, int last_action, int agent_id,
                                               const marl_agent_params* p, const float* obs, const float* last_onehot,
                                               const float* avail, const float* h_in, float* h_out,
                                               const marl_act_philox* philox, double eps, const int* gate,
                                               long long* action, float* onehot, float* q, void* stream) {
    ActPhilox ph;
    if (!philox_ok(philox, ph)) return MARL_EINVAL;
    return act_call<true, true>(n_envs, N, A, O, last_action, agent_id, p, obs, last_onehot, avail, h_in, h_out, nullptr,
                                nullptr, nullptr, nullptr, eps, gate, action, onehot, q, ph, stream);
}

namespace marl {
__global__ void philox_uniforms_kernel(unsigned long long seed, unsigned long long episode_base, int step, int n_envs,
                                       int N, double* out) {
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= (long long)n_envs * N) return;
    const int e = (int)(row / N), n = (int)(row - (long long)e * N);
    philox_act_uniforms(seed, episode_base + (unsigned long long)e, step, n, out[2 * row], out[2 * row + 1]);
}
}  // namespace marl

extern "C" int marl_philox_uniforms(unsigned long long seed, unsigned long long episode_base, int step, int n_envs, int N,
                                    double* out, void* stream) {
    if (n_envs < 0 || N <= 0 || step < 0 || !out || (long long)n_envs * N > 0x7fffffffLL) return MARL_EINVAL;
    const long long rows = (long long)n_envs * N;
    if (rows == 0) return MARL_OK;
    { ProfScope ps_("philox_uniforms_kernel", (cudaStream_t)stream);
      philox_uniforms_kernel<<<(int)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(seed, episode_base, step, n_envs,
                                                                                         N, out); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

extern "C" int marl_rollout_record(const marl_dims* d, int t, const marl_episode_f32* ep, const float* obs, const float* state,
                                   const float* avail, const long long* action, const float* onehot, const double* reward,
                                   const unsigned char* terminated, unsigned char* active, float* last, double* reward_sum,
                                   int* counters, int* active_host, void* stream) {
    if (!d || !ep || d->B < 0 || d->L <= 0 || d->N <= 0 || d->A <= 0 || d->O < 0 || d->S < 0 || t < 0 || t > d->L) return MARL_EINVAL;
    if (!ep->o || !ep->s || !ep->u || !ep->r || !ep->o_next || !ep->s_next || !ep->avail_u || !ep->avail_u_next ||
        !ep->u_onehot || !ep->padded || !ep->terminated)
        return MARL_EINVAL;
    if (!obs || !state || !avail || !active || !last || !reward_sum || !counters) return MARL_EINVAL;
    if (t > 0 && (!action || !onehot || !reward || !terminated)) return MARL_EINVAL;
    if (d->B == 0) return MARL_OK;
    RecArgs a{*d, t, *ep, obs, state, avail, action, onehot, reward, terminated, active, last, reward_sum, counters, active_host};
    { ProfScope ps_("rollout_record_kernel", (cudaStream_t)stream);
      rollout_record_kernel<<<(d->B + kRecWarps - 1) / kRecWarps, kRecWarps * 32, 0, (cudaStream_t)stream>>>(a); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}
