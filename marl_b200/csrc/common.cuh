// Shared device helpers for libmarl_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define MARL_H 64            // rnn_hidden_dim  (common/arguments.py:88)
#define MARL_G (3 * MARL_H)  // GRU gate width (r,z,n)

#define MARL_OK 0
#define MARL_EINVAL (-1)

#define MARL_LAUNCH_CHECK()                                   \
    do {                                                      \
        cudaError_t e__ = cudaGetLastError();                 \
        if (e__ != cudaSuccess) return (int)e__;              \
    } while (0)

#include <cstdlib>
#include <utility>

namespace marl {

constexpr int kNumSMs = 148;

// rnn_hidden_dim as a parameter struct carries it (marl_agent_params.hidden, marl_qtran_net_params.hidden): 0 means 64;
// -1 for a width the kernels do not serve (only 32, 64 and 128 are built)
inline int hidden_width(int hidden) {
    const int h = hidden ? hidden : MARL_H;
    return (h == 32 || h == MARL_H || h == 128) ? h : -1;
}

// ---- programmatic dependent launch ------------------------------------------------------------------------
// Kernels on the step's dependent chain start with pdl_enter(): wait until the grids they depend on have completed
// and flushed (a no-op when launched normally), then let the NEXT kernel of the stream be scheduled early -- its CTAs
// become resident and sit in their own pdl_enter() -- so that the ~2.5 us launch gap between two dependent kernels
// of the captured graph is hidden.  (Kernels whose grids span several waves trigger late, pdl_wait() ... pdl_trigger(),
// so that waiting dependents do not take SM residency from their own remaining CTAs.)  Nothing may touch global
// memory before the wait, and every CTA must pass it
// (even the ones that return early), otherwise completion of this grid would not imply completion of its predecessors.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// single-wave kernels: let the dependents become resident right away
__device__ __forceinline__ void pdl_enter() { pdl_wait(); pdl_trigger(); }
inline bool pdl_enabled() {
    static int on = -1;
    if (on < 0) { const char* e = getenv("MARL_B200_PDL"); on = (e && e[0] == '0') ? 0 : 1; }
    return on == 1;
}
// Early residency of the next kernel only pays in the latency-bound regime (a few hundred CTAs per launch); with
// many-wave grids the waiting CTAs take slots from the running kernel (measured: cfg 2 -4 %, cfg 3/4 +1.3..2.6 %).
// The operator entry points set the regime from their problem size before they launch.
inline bool& pdl_small_problem() { static bool v = true; return v; }
inline void pdl_scope(long long rows) { pdl_small_problem() = rows <= 65536; }
// <<<grid, block, smem, st>>> with the programmatic-stream-serialization attribute; only for kernels that call pdl_wait()
// prio < 0: launch-priority attribute (numerically lower = scheduled first), so that the one-CTA-per-SM recurrence
// kernels get their CTAs placed ahead of GEMM CTAs from sibling streams that became ready at the same moment
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl_prio(int prio, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_enabled() && pdl_small_problem()) ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (prio < 0) {
        attr[1].id = cudaLaunchAttributePriority;
        attr[1].val.priority = prio;
        cfg.numAttrs = 2;
    }
    return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}
// launch priority of the GEMM launches issued while a LinearPrio is alive (host calls are single-threaded)
inline int& linear_prio() { static int v = 0; return v; }
struct LinearPrio {
    int keep;
    explicit LinearPrio(int p) : keep(linear_prio()) { linear_prio() = p; }
    ~LinearPrio() { linear_prio() = keep; }
};
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    return launch_pdl_prio(0, kern, grid, block, smem, st, std::forward<Args>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// ------------------------------------------------------------------------------------------
// Linear-layer operand description shared by the forward / data-gradient / weight-gradient
// GEMM kernels.  The logical input row is the K-wide concatenation
//     [ x (K1 cols) | x2 (K2 cols, optionally shifted by `x2_shift` rows within a period) |
//       one-hot(m % onehot_mod) (onehot_mod cols) ]
// which is how the agent input [obs | last_action | agent_id] (share_params.py:84-112) and the
// QTRAN [hidden | action] / [state | encoding] concatenations are consumed without ever being
// materialised.  With onehot_z the one-hot column is the batched problem's index z instead: a
// launch over z = agent whose problem z holds the rows of agent z only (SeparatedMAC's input,
// share_params.py:467-495).
// ------------------------------------------------------------------------------------------
struct LinOperand {
    const float* x;   int ldx;  int K1;
    const float* x2;  int ldx2; int K2;
    int x2_shift;     // rows; element (m, K1+k) reads x2[m - shift] and is 0 when (m % x2_period) < shift
    int x2_period;
    int onehot_mod;   // 0 = none
    long long x_bs, x2_bs;   // blockIdx.z strides (batched problems)
    int onehot_z;     // 1: the hot column is z (k == z) rather than m % onehot_mod
};

__device__ __forceinline__ float lin_load(const LinOperand& a, int z, int m, int k) {
    if (k < a.K1) return __ldg(a.x + (long long)z * a.x_bs + (long long)m * a.ldx + k);
    k -= a.K1;
    if (k < a.K2) {
        int mm = m;
        if (a.x2_shift) {
            if ((m % a.x2_period) < a.x2_shift) return 0.0f;
            mm = m - a.x2_shift;
        }
        return __ldg(a.x2 + (long long)z * a.x2_bs + (long long)mm * a.ldx2 + k);
    }
    k -= a.K2;
    return (a.onehot_z ? z : m % a.onehot_mod) == k ? 1.0f : 0.0f;
}

__host__ __device__ __forceinline__ int lin_width(const LinOperand& a) { return a.K1 + a.K2 + a.onehot_mod; }

}  // namespace marl
