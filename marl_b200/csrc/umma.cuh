// Internal (non-ABI): operand fetchers, TF32 split and tcgen05 / mbarrier helpers shared by the tensor-core kernels
// (linear.cu, front.cu, tail.cu).
#pragma once
#include "linear.h"

namespace marl {

// ---- operand fetchers: one float4 (4 consecutive elements along the contiguous dim) per call ---------

// Operand described by a LinOperand: logical matrix [rows, width], contiguous along the column index.
struct OpLin {
    LinOperand o; int z; int rows; int width; bool vec; bool vec2;
    // everything that depends on the row only (pointers into the two sources, the one-hot column): computed once per
    // thread when the row is fixed for the whole k-loop -- the per-tile fetch is then a range test and a load
    struct Row { const float* xr; const float* x2r; int hot; bool valid; };
    __device__ __forceinline__ Row row(int i) const {
        Row rw{nullptr, nullptr, -1, i < rows};
        if (!rw.valid) return rw;
        if (o.x) rw.xr = o.x + (long long)z * o.x_bs + (long long)i * o.ldx;
        if (o.K2 > 0 && !(o.x2_shift && (i % o.x2_period) < o.x2_shift))
            rw.x2r = o.x2 + (long long)z * o.x2_bs + (long long)(i - o.x2_shift) * o.ldx2 - o.K1;
        if (o.onehot_mod) rw.hot = o.K1 + o.K2 + (o.onehot_z ? z : i % o.onehot_mod);
        return rw;
    }
    __device__ __forceinline__ float4 quad_at(const Row& rw, int r) const {   // elements (row, r..r+3)
        if (!rw.valid) return make_float4(0.f, 0.f, 0.f, 0.f);
        if (vec && r + 3 < o.K1) return __ldg(reinterpret_cast<const float4*>(rw.xr + r));
        if (vec2 && r >= o.K1 && r + 3 < o.K1 + o.K2)
            return rw.x2r ? __ldg(reinterpret_cast<const float4*>(rw.x2r + r)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float e[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int k = r + c;
            float val = 0.f;
            if (k < o.K1) val = __ldg(rw.xr + k);
            else if (k < o.K1 + o.K2) { if (rw.x2r) val = __ldg(rw.x2r + k); }
            else if (k == rw.hot) val = 1.0f;
            e[c] = val;
        }
        return make_float4(e[0], e[1], e[2], e[3]);
    }
    __device__ __forceinline__ float4 quad(int i, int r) const {   // elements (i, r..r+3)
        if (i >= rows) return make_float4(0.f, 0.f, 0.f, 0.f);
        if (vec && r + 3 < o.K1)
            return __ldg(reinterpret_cast<const float4*>(o.x + (long long)z * o.x_bs + (long long)i * o.ldx + r));
        if (vec2 && r >= o.K1 && r + 3 < o.K1 + o.K2) {
            int ii = i;
            if (o.x2_shift) {
                if ((i % o.x2_period) < o.x2_shift) return make_float4(0.f, 0.f, 0.f, 0.f);
                ii = i - o.x2_shift;
            }
            return __ldg(reinterpret_cast<const float4*>(o.x2 + (long long)z * o.x2_bs + (long long)ii * o.ldx2 + (r - o.K1)));
        }
        // ragged / virtual part: row-level work (shift test, agent id) once per quad
        const float* xr = o.x ? o.x + (long long)z * o.x_bs + (long long)i * o.ldx : nullptr;
        const bool x2_live = o.K2 > 0 && !(o.x2_shift && (i % o.x2_period) < o.x2_shift);
        const float* x2r = x2_live ? o.x2 + (long long)z * o.x2_bs + (long long)(i - o.x2_shift) * o.ldx2 - o.K1 : nullptr;
        const int hot = o.onehot_mod ? o.K1 + o.K2 + (o.onehot_z ? z : i % o.onehot_mod) : -1;
        float e[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int k = r + c;
            float val = 0.f;
            if (k < o.K1) val = __ldg(xr + k);
            else if (k < o.K1 + o.K2) { if (x2_live) val = __ldg(x2r + k); }
            else if (k == hot) val = 1.0f;
            e[c] = val;
        }
        return make_float4(e[0], e[1], e[2], e[3]);
    }
};

// Plain row-major matrix P[rows, cols] (ld), fetched along its contiguous (column) dimension.
struct OpMat {
    const float* p; int ld; int rows; int cols; bool vec;
    struct Row { const float* q; };      // row pointer (null beyond the matrix): hoisted out of the k-loop when the row is fixed
    __device__ __forceinline__ Row row(int r) const { return Row{r < rows ? p + (long long)r * ld : nullptr}; }
    __device__ __forceinline__ float4 quad_at(const Row& rw, int col) const {
        if (!rw.q) return make_float4(0.f, 0.f, 0.f, 0.f);
        const float* q = rw.q + col;
        if (vec && col + 3 < cols) return __ldg(reinterpret_cast<const float4*>(q));
        float4 v;
        v.x = col + 0 < cols ? __ldg(q + 0) : 0.f;
        v.y = col + 1 < cols ? __ldg(q + 1) : 0.f;
        v.z = col + 2 < cols ? __ldg(q + 2) : 0.f;
        v.w = col + 3 < cols ? __ldg(q + 3) : 0.f;
        return v;
    }
    __device__ __forceinline__ float4 quad(int row, int col) const {   // elements (row, col..col+3)
        if (row >= rows) return make_float4(0.f, 0.f, 0.f, 0.f);
        const float* q = p + (long long)row * ld + col;
        if (vec && col + 3 < cols) return __ldg(reinterpret_cast<const float4*>(q));
        float4 v;
        v.x = col + 0 < cols ? __ldg(q + 0) : 0.f;
        v.y = col + 1 < cols ? __ldg(q + 1) : 0.f;
        v.z = col + 2 < cols ? __ldg(q + 2) : 0.f;
        v.w = col + 3 < cols ? __ldg(q + 3) : 0.f;
        return v;
    }
};

// second-source 128-bit loads: x2 aligned, pitches and region starts multiples of 4 floats
__host__ __device__ __forceinline__ bool vec2_ok(const LinOperand& o) {
    return o.K2 >= 4 && o.x2 && (reinterpret_cast<uintptr_t>(o.x2) & 15) == 0 && (o.ldx2 & 3) == 0 &&
           (o.K1 & 3) == 0 && (o.K2 & 3) == 0 && (o.x2_bs & 3) == 0;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 64-bit shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp layout): start address, leading /
// stride byte offsets (all >> 4), version 1, no swizzle.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}

// Bounded wait on an mbarrier phase: a protocol bug traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    for (int spins = 0; !done; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (spins > (1 << 24)) __trap();
    }
}
// x = hi + lo with both halves ROUNDED to TF32 (cvt.rna): unbiased, unlike the truncation the tensor core
// applies to raw fp32 words, whose error grows linearly with the reduction length.
// (integer add + mask on the bit pattern = round to nearest, ties away, exactly what cvt.rna.tf32.f32 does for finite
// inputs; cvt itself runs on the quarter-rate conversion pipe and was measured to bound the split pass)
__device__ __forceinline__ float tf32_rna(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) { hi = tf32_rna(x); lo = tf32_rna(x - hi); }

}  // namespace marl
