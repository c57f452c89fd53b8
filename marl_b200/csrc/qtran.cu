// QTRAN-base joint networks: QtranQBase and QtranV (network/mixer.py:355-418) and the three QTRAN
// losses (algorithm/qtran_learner.py:103-152), forward + backward.
//
// Both networks share one shape -- a per-agent 2-layer encoder, a sum over agents, a 3-layer head on
// [state | encoding] -- so one "joint net" implementation serves both (Q: rows [hidden | action one-hot],
// V: rows [hidden]).  The second encoder layer is applied AFTER the sum over agents,
//     sum_n (W2 x_n + b2) = W2 (sum_n x_n) + N b2,
// which divides its cost by N; concatenations are never materialised (two-source GEMM operands).
#include "linear.h"
#include "forkjoin.h"
#include "../../include/marl_b200.h"
#include "profile.h"

namespace marl {

constexpr float kNegBigT = -9999999.0f;    // qtran_learner.py:106
constexpr float kNegEval = -999999.0f;     // qtran_learner.py:105

// es[m, :] = sum_n e1[m*N + n, :]
__global__ void __launch_bounds__(256) agent_sum_kernel(int M, int N, int D, const float* __restrict__ e1, float* __restrict__ es) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * D) return;
    const int m = (int)(i / D), c = (int)(i % D);
    float acc = 0.f;
    for (int n = 0; n < N; ++n) acc += e1[((long long)m * N + n) * D + c];
    es[i] = acc;
}

// de1[m*N + n, :] = des[m, :] * (e1 > 0)
__global__ void __launch_bounds__(256) agent_bcast_relu_kernel(int M, int N, int D, const float* __restrict__ des,
                                                              const float* __restrict__ e1, float* __restrict__ de1) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * N * D) return;
    const long long row = i / D; const int c = (int)(i % D);
    de1[i] = e1[i] > 0.f ? des[(row / N) * D + c] : 0.f;
}

__global__ void __launch_bounds__(256) qtran_select_kernel(int rows, int A, const float* __restrict__ q_evals,
    float* __restrict__ q_targets, const float* __restrict__ avail, const float* __restrict__ avail_next,
    const long long* __restrict__ u, float* __restrict__ oh_eval, float* __restrict__ oh_target,
    long long* __restrict__ opt_eval, float* __restrict__ q_max_eval, float* __restrict__ q_taken) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const long long o = (long long)i * A;
    int be = 0, bt = 0; float ve = 0.f, vt = 0.f;
    for (int a = 0; a < A; ++a) {
        const float e = (avail[o + a] == 0.0f) ? kNegEval : q_evals[o + a];          // qtran_learner.py:104-105
        if (a == 0 || e > ve) { ve = e; be = a; }
        float t = q_targets[o + a];
        if (avail_next[o + a] == 0.0f) { t = kNegBigT; q_targets[o + a] = t; }        // in place, :106
        if (a == 0 || t > vt) { vt = t; bt = a; }
    }
    for (int a = 0; a < A; ++a) {                                                     // :108-114
        oh_eval[o + a] = (a == be) ? 1.0f : 0.0f;
        oh_target[o + a] = (a == bt) ? 1.0f : 0.0f;
    }
    opt_eval[i] = be;
    q_max_eval[i] = ve;                                                               // :129
    q_taken[i] = q_evals[o + u[i]];                                                   // :143
}

__device__ __forceinline__ void block_add(float* out, const float* vals, int n) {
    __shared__ float red[4][32];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    for (int k = 0; k < n; ++k) { float v = warp_sum(vals[k]); if (l == 0) red[k][w] = v; }
    __syncthreads();
    if (w == 0)
        for (int k = 0; k < n; ++k) { float v = l < nw ? red[k][l] : 0.f; v = warp_sum(v); if (l == 0) atomicAdd(out + k, v); }
}

__global__ void __launch_bounds__(256) qtran_loss_kernel(int M, int N, int A, const float* jq, const float* jq_t,
    const float* jq_hat, const float* v, const float* q_max_eval, const float* q_taken, const long long* opt_eval,
    const long long* u, const float* avail, const float* r, const float* term, const float* padded, float gamma,
    float lam_opt, float lam_nopt, float* d_jq, float* d_v, float* dq, float* scalars, float* parts) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (m < M) {
        const float mask = 1.0f - padded[m];                                          // qtran_learner.py:85
        const float y = r[m] + gamma * jq_t[m] * (1.0f - term[m]);                    // :121
        const float td = (jq[m] - y) * mask;                                          // :122-123
        float so = 0.f, sn = 0.f;
        for (int n = 0; n < N; ++n) { so += q_max_eval[m * N + n]; sn += q_taken[m * N + n]; }   // :129, :144
        const float opt = (so - jq_hat[m] + v[m]) * mask;                             // :137-138
        float nopt = sn - jq[m] + v[m];                                               // :146
        nopt = fminf(nopt, 0.0f) * mask;                                              // :147-148
        acc[0] = td * td; acc[1] = opt * opt; acc[2] = nopt * nopt; acc[3] = mask;
        const float g_opt = 2.0f * mask * lam_opt * opt, g_nopt = 2.0f * mask * lam_nopt * nopt;
        d_jq[m] = 2.0f * mask * td;                       // joint_q is detached inside l_nopt (:146)
        d_v[m] = g_opt + g_nopt;
        for (int n = 0; n < N; ++n) {
            const long long o = ((long long)m * N + n) * A;
            const int oa = (int)opt_eval[m * N + n], ua = (int)u[m * N + n];
            const bool live = avail[o + oa] != 0.0f;      // a masked maximum is a constant: no gradient
            for (int c = 0; c < A; ++c) {
                float g = 0.f;
                if (c == oa && live) g += g_opt;
                if (c == ua) g += g_nopt;
                dq[o + c] = g;
            }
        }
    }
    block_add(parts, acc, 3);
    float two[2] = {acc[0] + lam_opt * acc[1] + lam_nopt * acc[2], acc[3]};
    __syncthreads();
    block_add(scalars, two, 2);
}

struct JointLayout { int N, S, H, Aenc, Din, qh; };

static LinOperand enc_input(const JointLayout& l, const float* hidden, const float* actions) {
    LinOperand in = plain_operand(hidden, l.H, l.H);
    if (l.Aenc) { in.x2 = actions; in.ldx2 = l.Aenc; in.K2 = l.Aenc; }
    return in;
}
static LinOperand head_input(const JointLayout& l, const float* s, const float* enc) {
    LinOperand in = plain_operand(s, l.S, l.S);
    in.x2 = enc; in.ldx2 = l.Din; in.K2 = l.Din;
    return in;
}

static int joint_fwd(int M, const JointLayout& l, const marl_qtran_net_params* p, const float* s, const float* hidden,
                     const float* actions, const marl_qtran_net_ws* ws, float* out, cudaStream_t st) {
    int rc;
    const int rows = M * l.N;
    LinearFwd f{};
    f.in = enc_input(l, hidden, actions); f.w = p->we1; f.ldw = l.Din; f.bias = p->be1;
    f.y = ws->e1; f.ldy = l.Din; f.M = rows; f.N = l.Din; f.relu = 1; f.batch = 1;
    if ((rc = linear_fwd(f, st))) return rc;
    {
        const long long n = (long long)M * l.Din;
        ProfScope ps_("agent_sum_kernel", st);
        agent_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(M, l.N, l.Din, ws->e1, ws->es);
    }
    MARL_LAUNCH_CHECK();
    LinearFwd f2{};
    f2.in = plain_operand(ws->es, l.Din, l.Din); f2.w = p->we2; f2.ldw = l.Din; f2.bias = p->be2; f2.bias_mul = (float)l.N;
    f2.y = ws->enc; f2.ldy = l.Din; f2.M = M; f2.N = l.Din; f2.batch = 1;
    if ((rc = linear_fwd(f2, st))) return rc;
    LinearFwd h0{};
    h0.in = head_input(l, s, ws->enc); h0.w = p->w0; h0.ldw = l.S + l.Din; h0.bias = p->b0;
    h0.y = ws->a1; h0.ldy = l.qh; h0.M = M; h0.N = l.qh; h0.relu = 1; h0.batch = 1;
    if ((rc = linear_fwd(h0, st))) return rc;
    LinearFwd h2{};
    h2.in = plain_operand(ws->a1, l.qh, l.qh); h2.w = p->w2; h2.ldw = l.qh; h2.bias = p->b2;
    h2.y = ws->a2; h2.ldy = l.qh; h2.M = M; h2.N = l.qh; h2.relu = 1; h2.batch = 1;
    if ((rc = linear_fwd(h2, st))) return rc;
    LinearFwd h4{};
    h4.in = plain_operand(ws->a2, l.qh, l.qh); h4.w = p->w4; h4.ldw = l.qh; h4.bias = p->b4;
    h4.y = out; h4.ldy = 1; h4.M = M; h4.N = 1; h4.batch = 1;
    return linear_fwd(h4, st);
}

static int joint_bwd(int M, const JointLayout& l, const marl_qtran_net_params* p, const float* s, const float* hidden,
                     const float* actions, const marl_qtran_net_ws* ws, const float* dout, const marl_qtran_net_ws* dws,
                     float* dhidden, int accumulate_dhidden, const marl_qtran_net_grads* g, cudaStream_t st) {
    int rc;
    const int rows = M * l.N;
    // The data gradients are the dependent chain; each weight gradient only reads the dy its layer already has, so it goes to a
    // forked lane (one side stream, forked anew behind every producer) and runs beside the rest of the chain -- the eager timeline
    // of config 4 (profiles/r2c_cfg4_timeline.txt) had 212 us of weight gradients between 164 us of chain per network.
    ForkJoin fj(st, 2);
    auto lane = [&]() { ForkJoin f(st, 2); return f.lane(1); };      // behind everything queued on `st` so far
    {   // head layer 4
        LinearWgrad w{}; w.dy = dout; w.lddy = 1; w.in = plain_operand(ws->a2, l.qh, l.qh);
        w.dw = g->w4; w.ldw = l.qh; w.db = g->b4; w.M = M; w.N = 1; w.batch = 1;
        if ((rc = linear_wgrad(w, lane()))) return rc;
        LinearDgrad d{}; d.dy = dout; d.lddy = 1; d.w = p->w4; d.ldw = l.qh; d.dx = dws->a2; d.lddx = l.qh;
        d.relu_src = ws->a2; d.ldrs = l.qh; d.M = M; d.N = 1; d.K = l.qh; d.batch = 1;
        if ((rc = linear_dgrad(d, st))) return rc;
    }
    {   // head layer 2
        LinearWgrad w{}; w.dy = dws->a2; w.lddy = l.qh; w.in = plain_operand(ws->a1, l.qh, l.qh);
        w.dw = g->w2; w.ldw = l.qh; w.db = g->b2; w.M = M; w.N = l.qh; w.batch = 1;
        if ((rc = linear_wgrad(w, lane()))) return rc;
        LinearDgrad d{}; d.dy = dws->a2; d.lddy = l.qh; d.w = p->w2; d.ldw = l.qh; d.dx = dws->a1; d.lddx = l.qh;
        d.relu_src = ws->a1; d.ldrs = l.qh; d.M = M; d.N = l.qh; d.K = l.qh; d.batch = 1;
        if ((rc = linear_dgrad(d, st))) return rc;
    }
    {   // head layer 0 on [s | enc]: weights for both parts, data gradient only for the encoding
        LinearWgrad w{}; w.dy = dws->a1; w.lddy = l.qh; w.in = head_input(l, s, ws->enc);
        w.dw = g->w0; w.ldw = l.S + l.Din; w.db = g->b0; w.M = M; w.N = l.qh; w.batch = 1;
        if ((rc = linear_wgrad(w, lane()))) return rc;
        LinearDgrad d{}; d.dy = dws->a1; d.lddy = l.qh; d.w = p->w0; d.ldw = l.S + l.Din; d.w_col0 = l.S;
        d.dx = dws->enc; d.lddx = l.Din; d.M = M; d.N = l.qh; d.K = l.Din; d.batch = 1;
        if ((rc = linear_dgrad(d, st))) return rc;
    }
    {   // encoder layer 2 (applied to the agent sum; bias counted N times)
        LinearWgrad w{}; w.dy = dws->enc; w.lddy = l.Din; w.in = plain_operand(ws->es, l.Din, l.Din);
        w.dw = g->we2; w.ldw = l.Din; w.db = g->be2; w.db_mul = (float)l.N; w.M = M; w.N = l.Din; w.batch = 1;
        if ((rc = linear_wgrad(w, lane()))) return rc;
        LinearDgrad d{}; d.dy = dws->enc; d.lddy = l.Din; d.w = p->we2; d.ldw = l.Din; d.dx = dws->es; d.lddx = l.Din;
        d.M = M; d.N = l.Din; d.K = l.Din; d.batch = 1;
        if ((rc = linear_dgrad(d, st))) return rc;
    }
    {
        const long long n = (long long)rows * l.Din;
        ProfScope ps_("agent_bcast_relu_kernel", st);
        agent_bcast_relu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(M, l.N, l.Din, dws->es, ws->e1, dws->e1);
    }
    MARL_LAUNCH_CHECK();
    {   // encoder layer 1 on [hidden | actions]
        LinearWgrad w{}; w.dy = dws->e1; w.lddy = l.Din; w.in = enc_input(l, hidden, actions);
        w.dw = g->we1; w.ldw = l.Din; w.db = g->be1; w.M = rows; w.N = l.Din; w.batch = 1;
        if ((rc = linear_wgrad(w, lane()))) return rc;
        if (dhidden) {
            LinearDgrad d{}; d.dy = dws->e1; d.lddy = l.Din; d.w = p->we1; d.ldw = l.Din; d.w_col0 = 0;
            d.dx = dhidden; d.lddx = l.H; d.M = rows; d.N = l.Din; d.K = l.H; d.accumulate = accumulate_dhidden; d.batch = 1;
            if ((rc = linear_dgrad(d, st))) return rc;
        }
    }
    fj.join();
    return MARL_OK;
}

static bool net_ok(const marl_qtran_net_params* p, const marl_qtran_net_ws* ws) {
    return p && ws && p->we1 && p->be1 && p->we2 && p->be2 && p->w0 && p->b0 && p->w2 && p->b2 && p->w4 && p->b4 &&
           ws->e1 && ws->es && ws->enc && ws->a1 && ws->a2;
}

}  // namespace marl

using namespace marl;

extern "C" int marl_qtran_net_fwd(int M, int N, int S, int A_enc, int qh, const marl_qtran_net_params* p, const float* s,
                                  const float* hidden, const float* actions, const marl_qtran_net_ws* ws, float* out,
                                  void* stream) {
    if (M < 0 || N < 1 || S < 1 || A_enc < 0 || qh < 1 || !net_ok(p, ws) || !s || !hidden || !out) return MARL_EINVAL;
    if (A_enc > 0 && !actions) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    const int H = hidden_width(p->hidden);
    if (H < 0) return MARL_EINVAL;
    const JointLayout l{N, S, H, A_enc, H + A_enc, qh};
    return joint_fwd(M, l, p, s, hidden, actions, ws, out, (cudaStream_t)stream);
}

extern "C" int marl_qtran_net_bwd(int M, int N, int S, int A_enc, int qh, const marl_qtran_net_params* p, const float* s,
                                  const float* hidden, const float* actions, const marl_qtran_net_ws* ws, const float* dout,
                                  const marl_qtran_net_ws* dws, float* dhidden, int accumulate_dhidden,
                                  const marl_qtran_net_grads* g, void* stream) {
    if (M < 0 || N < 1 || S < 1 || A_enc < 0 || qh < 1 || !net_ok(p, ws) || !s || !hidden || !dout || !dws || !g)
        return MARL_EINVAL;
    if (!dws->e1 || !dws->es || !dws->enc || !dws->a1 || !dws->a2) return MARL_EINVAL;
    if (A_enc > 0 && !actions) return MARL_EINVAL;
    if (M == 0) return MARL_OK;
    const int H = hidden_width(p->hidden);
    if (H < 0) return MARL_EINVAL;
    const JointLayout l{N, S, H, A_enc, H + A_enc, qh};
    return joint_bwd(M, l, p, s, hidden, actions, ws, dout, dws, dhidden, accumulate_dhidden, g, (cudaStream_t)stream);
}

extern "C" int marl_qtran_select(const marl_dims* d, const float* q_evals, float* q_targets, const float* avail_u,
                                 const float* avail_u_next, const long long* u, float* opt_onehot_eval,
                                 float* opt_onehot_target, long long* opt_action_eval, float* q_max_eval, float* q_taken,
                                 void* stream) {
    if (!d || !q_evals || !q_targets || !avail_u || !avail_u_next || !u || !opt_onehot_eval || !opt_onehot_target ||
        !opt_action_eval || !q_max_eval || !q_taken)
        return MARL_EINVAL;
    const int rows = d->B * d->L * d->N;
    if (rows <= 0) return MARL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    { ProfScope ps_("qtran_select_kernel", st);
      qtran_select_kernel<<<(rows + 255) / 256, 256, 0, st>>>(rows, d->A, q_evals, q_targets, avail_u, avail_u_next, u,
          opt_onehot_eval, opt_onehot_target, opt_action_eval, q_max_eval, q_taken); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

extern "C" int marl_qtran_losses_fwd_bwd(const marl_dims* d, const float* joint_q, const float* joint_q_target,
                                         const float* joint_q_hat, const float* v, const float* q_max_eval,
                                         const float* q_taken, const long long* opt_action_eval, const long long* u,
                                         const float* avail_u, const float* r, const float* terminated, const float* padded,
                                         float gamma, float lambda_opt, float lambda_nopt, float* d_joint_q, float* d_v,
                                         float* dq, float* scalars, float* loss_parts, void* stream) {
    if (!d || !joint_q || !joint_q_target || !joint_q_hat || !v || !q_max_eval || !q_taken || !opt_action_eval || !u ||
        !avail_u || !r || !terminated || !padded || !d_joint_q || !d_v || !dq || !scalars || !loss_parts)
        return MARL_EINVAL;
    const int M = d->B * d->L;
    if (M <= 0) return MARL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    { ProfScope ps_("qtran_loss_kernel", st);
      qtran_loss_kernel<<<(M + 255) / 256, 256, 0, st>>>(M, d->N, d->A, joint_q, joint_q_target, joint_q_hat, v, q_max_eval,
          q_taken, opt_action_eval, u, avail_u, r, terminated, padded, gamma, lambda_opt, lambda_nopt, d_joint_q, d_v, dq,
          scalars, loss_parts); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}
