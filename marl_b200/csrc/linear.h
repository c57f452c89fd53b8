// Internal (non-ABI) dense-layer primitives used by the operator files.
#pragma once
#include "common.cuh"

namespace marl {

// y[M,N] (+)= act( in[M,K] . w[N,K]^T + bias[N] )        (nn.Linear convention: w is [out, in])
struct LinearFwd {
    LinOperand in;
    const float* w;    int ldw;  long long w_bs;
    const float* bias;           long long b_bs;   // nullable
    float* y;          int ldy;  long long y_bs;
    int M, N;
    float bias_mul;   // bias is added as bias_mul * bias (0 means 1): sum over agents of a per-agent Linear
    int relu;         // apply max(0, .) in the epilogue
    int accumulate;   // y += result instead of y = result
    int batch;        // independent problems over blockIdx.z (operands advance by *_bs)
};

// dx[M,K] (+)= ( dy[M,N] . w[N, col0:col0+K] ) * (relu_src[M,K] > 0)
struct LinearDgrad {
    const float* dy;   int lddy; long long dy_bs;
    const float* w;    int ldw;  long long w_bs;  int w_col0;
    float* dx;         int lddx; long long dx_bs;
    const float* relu_src; int ldrs; long long rs_bs;   // nullable
    int M, N, K;
    int accumulate;
    int batch;
    // optional: the weight slice already transposed, wt[k, n] = w[n, w_col0 + k] (row pitch ldwt) -- both operands are then
    // contiguous along the reduction and take the 128-bit staging path (transpose_weights); batch must be 1
    const float* wt; int ldwt;
};

// dw[N, 0:K] += dy[M,N]^T . in[M,K] ;  db[N] += colsum(dy)   (atomic split over M)
struct LinearWgrad {
    const float* dy;   int lddy; long long dy_bs;
    LinOperand in;
    float* dw;         int ldw;  long long dw_bs;
    float* db;                   long long db_bs;   // nullable
    float db_mul;     // db += db_mul * colsum(dy) (0 means 1)
    int M, N;
    int batch;
};

// split weight gradients meet in a fixed-order second stage (bitwise reproducible) instead of atomics
bool deterministic_wgrad();
void set_deterministic_wgrad(int on);

// wt[k, n] = w[n, col0 + k] for n < N, k < K (one small launch); wt pitch = N rounded up to 4 floats
int transpose_weights(const float* w, int ldw, int col0, int N, int K, float* wt, cudaStream_t st);
inline int transposed_pitch(int N) { return (N + 3) & ~3; }
// tma = false: the register-staged kernels of this file even when the TMA back end (tgemm.cu) is on and would take the operands
int linear_fwd(const LinearFwd& a, cudaStream_t st, bool tma = true);
int linear_dgrad(const LinearDgrad& a, cudaStream_t st, bool tma = true);
int linear_wgrad(const LinearWgrad& a, cudaStream_t st, bool tma = true);

inline LinOperand plain_operand(const float* x, int ldx, int K, long long bs = 0) {
    LinOperand o{};
    o.x = x; o.ldx = ldx; o.K1 = K; o.x_bs = bs;
    o.x2 = nullptr; o.ldx2 = 0; o.K2 = 0; o.x2_shift = 0; o.x2_period = 1; o.onehot_mod = 0; o.x2_bs = 0; o.onehot_z = 0;
    return o;
}

}  // namespace marl
