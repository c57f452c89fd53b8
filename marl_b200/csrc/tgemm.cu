// TMA-fed, warp-specialised, persistent tcgen05 GEMM (3xTF32) for the dense layers and their autograd duals.
//
// Why a second GEMM kernel: the register-staged kernels of linear.cu spend their time in LDG -> split -> (scalar,
// transposing) STS sequences between CTA-wide barriers (profiles/README.md, "GEMM investigation").  Here
//   * operand tiles arrive by TMA (cp.async.bulk.tensor, 128-byte swizzle) straight in the layout the tensor core
//     reads: K-major operands as SWIZZLE_128B boxes of {32 floats, rows}; MN-major operands (the weight gradient
//     reduces over the ROWS of both of its row-major operands, the data gradient over the rows of W) as
//     SWIZZLE_128B_ATOM_32B boxes of {32 floats, 32 k-rows} described by a SWIZZLE_128B_BASE32B matrix descriptor --
//     no transposing stores anywhere (layouts validated with tools/micro/tma_probe.cu);
//   * four converter warps make ONE element-wise pass over a landed stage, in place: x -> hi = rna_tf32(x) (written
//     back) and lo = rna_tf32(x - hi) (second buffer, same swizzled offsets), then hand the stage to the MMA warp
//     through an mbarrier; one elected thread issues lo.hi + hi.lo + hi.hi per k8 step (tcgen05.mma kind::tf32);
//   * accumulators live in TMEM, double-buffered when they fit, so that four epilogue warps drain tile i
//     (tcgen05.ld -> bias / ReLU / mask -> global) while tile i+1 is loaded, converted and multiplied;
//   * one launch runs a GROUP of independent problems over persistent CTAs (one per SM);
//   * weight gradients are split over the reduction; every split writes its tile to a scratch arena and a second,
//     deterministic stage adds the splits in a fixed order (no atomics: run-to-run identical gradients).  The bias
//     gradient is a free extra row: a column of ones is written into the (padded) `in^T` operand.
//
// Replaces the cuBLAS addmm calls behind nn.Linear (network/q_network.py:17,20; network/mixer.py:45-55,117-145,
// 200-206,365-375,399-409) and their autograd duals whenever the operands are TMA-addressable (16-byte aligned base,
// row pitch a multiple of 16 bytes); everything else stays on linear.cu.
#include "tgemm.h"
#include "profile.h"
#include "../../include/marl_b200.h"
#include <cstring>
#include <cstdio>

namespace marl {

constexpr int TG_BM = 128, TG_BK = 32;
constexpr int TG_A_BYTES = TG_BM * TG_BK * 4;           // one raw A stage (16 KB); its lo copy follows
constexpr int TG_B_OFF = 2 * TG_A_BYTES;
constexpr int TG_THREADS = 320;                         // warp 0: TMA, warp 1: MMA, warps 2-5: converters, warps 6-9: epilogue
constexpr int TG_CVT0 = 64, TG_EPI0 = 192, TG_ROLE = 128;
constexpr int TG_MAX_STAGES = 6;
constexpr int TG_RING_BYTES = 188 * 1024;
constexpr int TG_TMEM_COLS = 512;

__device__ __forceinline__ uint32_t tg_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tg_mbar_init(uint64_t* b, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tg_u32(b)), "r"(count)); }
__device__ __forceinline__ void tg_mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tg_u32(b)) : "memory"); }
__device__ __forceinline__ void tg_mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tg_u32(b)), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void tg_mbar_wait(uint64_t* b, uint32_t parity) {
    uint32_t done = 0;
    for (int spins = 0; !done; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(tg_u32(b)), "r"(parity) : "memory");
        if (spins > (1 << 26)) __trap();
    }
}
__device__ __forceinline__ void tg_tma_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(tg_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(tg_u32(bar)) : "memory");
}
// matrix descriptor: start, LBO, SBO (>> 4), version 1, layout 2 = SWIZZLE_128B (K-major), 1 = SWIZZLE_128B_BASE32B (MN-major fp32)
__device__ __forceinline__ uint64_t tg_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
__device__ __forceinline__ uint64_t tg_op_desc(uint32_t tile, int mn, int k8) {
    // K-major: +32 B per k8 inside the 128-byte swizzle row, 8-row groups 1024 B apart.
    // MN-major: 8 k-rows = 1024 B per k8, 4-row atoms 512 B apart, 32-wide MN boxes 4096 B apart.
    return mn ? tg_desc(tile + (uint32_t)k8 * 1024u, 4096u, 512u, 1u) : tg_desc(tile + (uint32_t)k8 * 32u, 16u, 1024u, 2u);
}
__device__ __forceinline__ void tg_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tg_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tg_u32(bar)) : "memory");
}
// explicit state spaces (see the epilogue): no "memory" clobber, so that shared-memory loads may move across them
__device__ __forceinline__ void tg_st_global(float* p, float v) { asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v)); }
__device__ __forceinline__ float tg_ld_global(const float* p) { float v; asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v; }
__device__ __forceinline__ float tg_ldg_nc(const float* p) { float v; asm("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v; }
__device__ __forceinline__ float tg_rna(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

// byte offset of element (row r, column c) inside a landed tile
__device__ __forceinline__ uint32_t tg_off_k(int r, int c) {        // K-major tile: r = tile row, c = k (0..31)
    return (uint32_t)r * 128u + ((((uint32_t)c >> 2) ^ ((uint32_t)r & 7u)) << 4) + ((uint32_t)c & 3u) * 4u;
}
__device__ __forceinline__ uint32_t tg_off_mn(int k, int c) {       // MN-major tile: k = k-row (0..31), c = MN index (0..127)
    const uint32_t box = (uint32_t)c >> 5, cc = (uint32_t)c & 31u;
    return box * 4096u + (uint32_t)k * 128u + (((cc >> 3) ^ ((uint32_t)k & 3u)) << 5) + (cc & 7u) * 4u;
}

struct TGItem { int pi, m0, n0, kb0, kb1, local; };

// Optional phase trace of CTA 0 (MARL_TGEMM_TRACE=1 + marl_tgemm_trace_dump): (tag, clock64) pairs, 512 per role.
__device__ long long* g_tg_trace = nullptr;
static long long* g_trace_host = nullptr;          // the same buffer for kernels of other files (passed as an argument)
long long* trace_buffer() { return g_trace_host; }
#define TG_STAMP(role, tag)                                                                                   \
    do {                                                                                                      \
        if (trace && tn < 255) { trace[(role) * 512 + 2 * tn] = (tag); trace[(role) * 512 + 2 * tn + 1] = clock64(); ++tn; } \
    } while (0)

__device__ __forceinline__ TGItem tg_decode(const TGScalars* sp, int n, int item) {
    int pi = 0;
    while (pi + 1 < n && item >= sp[pi + 1].item0) ++pi;
    const TGScalars& p = sp[pi];
    TGItem it;
    it.pi = pi; it.local = item - p.item0;
    int l = it.local;
    const int mt = l % p.m_tiles; l /= p.m_tiles;
    const int nt = l % p.n_tiles; const int ks = l / p.n_tiles;
    it.m0 = mt * TG_BM; it.n0 = nt * p.BN;
    it.kb0 = ks * p.kb_per_split; it.kb1 = min(p.kb_total, it.kb0 + p.kb_per_split);
    return it;
}

__global__ void __launch_bounds__(TG_THREADS, 1) tgemm_kernel(const __grid_constant__ TGGroup g) {
    extern __shared__ unsigned char tg_smem_raw[];
    __shared__ uint64_t bar_full[TG_MAX_STAGES], bar_cvt[TG_MAX_STAGES], bar_empty[TG_MAX_STAGES], bar_accf[2], bar_acce[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(1024) float epi_stage[4][2 * 1024];       // per epilogue warp: two 32 x 32 blocks (TMA-store double buffer; the
                                                                     // st.global paths use the pair as one pitch-36 buffer)
    unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tg_smem_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    __shared__ TGScalars sp[TG_MAXP];
    const int S = g.n_stages, np = g.n;
    {
        // cooperative word copy of the problem scalars: parameter bank -> shared memory
        constexpr int W = sizeof(TGScalars) / 4;
        for (int i = tid; i < np * W; i += TG_THREADS)
            reinterpret_cast<uint32_t*>(sp)[i] = reinterpret_cast<const uint32_t*>(&g.p[i / W].s)[i % W];
    }
    if (tid == 0) {
        for (int s = 0; s < S; ++s) { tg_mbar_init(&bar_full[s], 1); tg_mbar_init(&bar_cvt[s], TG_ROLE); tg_mbar_init(&bar_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { tg_mbar_init(&bar_accf[b], 1); tg_mbar_init(&bar_acce[b], TG_ROLE); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int i = 0; i < g.n; ++i) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&g.p[i].mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&g.p[i].mapB) : "memory");
            if (g.p[i].s.out_tma) asm volatile("prefetch.tensormap [%0];" ::"l"(&g.p[i].mapOut) : "memory");
        }
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tg_u32(&tmem_base_s)), "r"(TG_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    long long* trace = (blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 6)) ? g_tg_trace : nullptr;
    int tn = 0;
    if (trace && warp == 0) { trace[2047] = 0; }
    pdl_wait();                                   // everything above overlaps the tail of the producing kernel

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int rit = 0;
            for (int item = blockIdx.x; item < g.total_items; item += gridDim.x) {
                const TGItem it = tg_decode(sp, np, item);
                const TGScalars p = sp[it.pi];      // by value: registers, not re-read after every store / asm
                const uint32_t tx = (uint32_t)TG_A_BYTES + (p.b_ptr ? 0u : (uint32_t)p.BN * 128u);
                for (int kb = it.kb0; kb < it.kb1; ++kb, ++rit) {
                    const int s = rit % S;
                    tg_mbar_wait(&bar_empty[s], (uint32_t)(((rit / S) & 1) ^ 1));
                    TG_STAMP(0, rit);
                    unsigned char* st = ring + (size_t)s * g.stage_bytes;
                    tg_mbar_expect_tx(&bar_full[s], tx);
                    const int k0 = kb * TG_BK;
                    if (!p.a_mn) tg_tma_2d(st, &g.p[it.pi].mapA, k0, it.m0, &bar_full[s]);
                    else
                        for (int j = 0; j < 4; ++j) tg_tma_2d(st + j * 4096, &g.p[it.pi].mapA, it.m0 + 32 * j, k0 - p.a_row_shift, &bar_full[s]);
                    if (!p.b_ptr) {
                        if (!p.b_mn) tg_tma_2d(st + TG_B_OFF, &g.p[it.pi].mapB, k0, it.n0, &bar_full[s]);
                        else
                            for (int j = 0; j < p.BN / 32; ++j) tg_tma_2d(st + TG_B_OFF + j * 4096, &g.p[it.pi].mapB, it.n0 + 32 * j, k0, &bar_full[s]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            int rit = 0, seq = 0;
            const bool dbg_nomma = (g.debug & 4) != 0;
            const int total_items = g.total_items, n_bufs = g.n_bufs, cols_per_buf = g.cols_per_buf, stage_bytes = g.stage_bytes;
            for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++seq) {
                const TGItem it = tg_decode(sp, np, item);
                const TGScalars p = sp[it.pi];      // by value: registers, not re-read after every store / asm
                const int buf = seq % g.n_bufs;
                tg_mbar_wait(&bar_acce[buf], (uint32_t)(((seq / g.n_bufs) & 1) ^ 1));      // the epilogue has drained this buffer
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t acc = tmem + (uint32_t)(buf * g.cols_per_buf);
                const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)p.a_mn << 15) | ((uint32_t)p.b_mn << 16) |
                                       ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(TG_BM >> 4) << 24);
                const uint32_t blo = (uint32_t)p.BN * 128u;
                int step = 0;
                for (int kb = it.kb0; kb < it.kb1; ++kb, ++rit) {
                    const int s = rit % S;
                    tg_mbar_wait(&bar_cvt[s], (uint32_t)((rit / S) & 1));
                    TG_STAMP(1, rit);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a0 = tg_u32(ring + (size_t)s * g.stage_bytes), b0 = a0 + TG_B_OFF;
#pragma unroll
                    for (int j = 0; j < 4 && !dbg_nomma; ++j, ++step) {
                        const uint64_t ah = tg_op_desc(a0, p.a_mn, j), al = tg_op_desc(a0 + TG_A_BYTES, p.a_mn, j);
                        const uint64_t bh = tg_op_desc(b0, p.b_mn, j), bl = tg_op_desc(b0 + blo, p.b_mn, j);
                        if (p.merge_corr) {
                            tg_mma(acc, al, bh, idesc, step ? 1u : 0u);
                            tg_mma(acc, ah, bl, idesc, 1u);
                            tg_mma(acc, ah, bh, idesc, 1u);
                        } else {
                            tg_mma(acc + (uint32_t)(p.nmain * p.BN), al, bh, idesc, step ? 1u : 0u);      // corrections
                            tg_mma(acc + (uint32_t)(p.nmain * p.BN), ah, bl, idesc, 1u);
                            tg_mma(acc + (uint32_t)((step % p.nmain) * p.BN), ah, bh, idesc, step >= p.nmain ? 1u : 0u);
                        }
                    }
                    tg_commit(&bar_empty[s]);             // stage free once these MMAs have read it
                    TG_STAMP(1, 1000 + rit);
                }
                tg_commit(&bar_accf[buf]);                // accumulators complete
            }
        }
    } else if (warp < 6) {
        // ================= converters: raw fix-ups, then x -> (hi in place, lo) =================
        const int ct = tid - TG_CVT0;
        int rit = 0;
        for (int item = blockIdx.x; item < g.total_items; item += gridDim.x) {
            const TGItem it = tg_decode(sp, np, item);
            const TGScalars p = sp[it.pi];      // by value: registers, not re-read after every store / asm
            const bool hooks = p.fill_on || p.a_row_shift || p.b_ptr;
            for (int kb = it.kb0; kb < it.kb1; ++kb, ++rit) {
                const int s = rit % S;
                unsigned char* st = ring + (size_t)s * g.stage_bytes;
                tg_mbar_wait(&bar_full[s], (uint32_t)((rit / S) & 1));
                TG_STAMP(2, rit);
                const int k0 = kb * TG_BK;
                if (hooks) {
                    if (p.a_row_shift) {
                        // rows of the shifted operand that would reach across an episode start are zero (h_{-1} = 0)
                        const int kr = ct >> 2, box = ct & 3;
                        if (((k0 + kr) % p.a_row_period) < p.a_row_shift) {
                            float4* d = reinterpret_cast<float4*>(st + box * 4096 + kr * 128);
#pragma unroll
                            for (int e = 0; e < 8; ++e) d[e] = make_float4(0.f, 0.f, 0.f, 0.f);
                        }
                        if (p.fill_on) asm volatile("bar.sync 1, %0;" ::"n"(TG_ROLE) : "memory");     // the ones column goes on top
                    }
                    if (p.fill_on) {
                        // one data row per thread at a time: the row's predicates are computed once, its values are
                        // fetched as a batch of independent loads and only then stored (a load -> store -> load chain
                        // through the generic store serialises one L2 latency per element)
                        const int W = p.fill_A + p.fill_N + p.fill_ones;
                        const bool mn = p.a_mn && p.fill_on == 1;
                        const int f0 = mn ? it.m0 : k0, fspan = mn ? TG_BM : TG_BK;
                        const int f_lo = max(p.fill_col0, f0), f_hi = min(p.fill_col0 + W, f0 + fspan);
                        const int R = mn ? TG_BK : (p.fill_on == 2 ? p.BN : TG_BM);
                        const int r0 = mn ? k0 : (p.fill_on == 2 ? it.n0 : it.m0);
                        unsigned char* tile = st + (p.fill_on == 2 ? TG_B_OFF : 0);
                        // MN-major tiles hold only 32 data rows: four threads share a row and interleave its features
                        const int lanes_per_row = mn ? TG_ROLE / TG_BK : 1;
                        const int rsub = mn ? ct / TG_BK : 0;
                        for (int r = mn ? ct % TG_BK : ct; r < R && f_lo < f_hi; r += mn ? TG_BK : TG_ROLE) {
                            const int row = r0 + r;
                            const bool live = row < p.fill_rows && !(p.fill_shift && (row % p.fill_period) < p.fill_shift);
                            const int id = p.fill_N ? row % p.fill_N : 0;
                            const float* oh = p.fill_onehot + (long long)(row - p.fill_shift) * p.fill_A - p.fill_col0;
                            for (int fb = f_lo + rsub; fb < f_hi; fb += 8 * lanes_per_row) {
                                float v[8];
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    const int f = fb + e * lanes_per_row, fr = f - p.fill_col0;
                                    v[e] = 0.f;
                                    if (f < f_hi) {
                                        if (fr < p.fill_A) { if (live) v[e] = __ldg(oh + f); }
                                        else if (fr < p.fill_A + p.fill_N) v[e] = (id == fr - p.fill_A) ? 1.f : 0.f;
                                        else v[e] = 1.f;
                                    }
                                }
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    const int f = fb + e * lanes_per_row;
                                    if (f < f_hi) *reinterpret_cast<float*>(tile + (mn ? tg_off_mn(r, f - f0) : tg_off_k(r, f - f0))) = v[e];
                                }
                            }
                        }
                    }
                    if (p.b_ptr) {
                        // B = dy gathered from global (row pitch not TMA-addressable), one 32-wide box
                        float v[8];
#pragma unroll
                        for (int l = 0; l < 8; ++l) {
                            const int idx = ct + TG_ROLE * l, kr = idx >> 5, c = idx & 31, row = k0 + kr, n = it.n0 + c;
                            v[l] = (row < p.Kd && n < p.Nd) ? __ldg(p.b_ptr + (long long)row * p.ldb + n) : 0.f;
                        }
#pragma unroll
                        for (int l = 0; l < 8; ++l) {
                            const int idx = ct + TG_ROLE * l;
                            *reinterpret_cast<float*>(st + TG_B_OFF + tg_off_mn(idx >> 5, idx & 31)) = v[l];
                        }
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(TG_ROLE) : "memory");
                }
                if (!(g.debug & 2)) {
                    float4* a4 = reinterpret_cast<float4*>(st);
                    float4* l4 = reinterpret_cast<float4*>(st + TG_A_BYTES);
                    float4 v[8];
#pragma unroll
                    for (int l = 0; l < 8; ++l) v[l] = a4[ct + TG_ROLE * l];
#pragma unroll
                    for (int l = 0; l < 8; ++l) {
                        const float4 h = make_float4(tg_rna(v[l].x), tg_rna(v[l].y), tg_rna(v[l].z), tg_rna(v[l].w));
                        a4[ct + TG_ROLE * l] = h;
                        l4[ct + TG_ROLE * l] = make_float4(tg_rna(v[l].x - h.x), tg_rna(v[l].y - h.y), tg_rna(v[l].z - h.z), tg_rna(v[l].w - h.w));
                    }
                }
                if (!(g.debug & 2)) {
                    float4* b4 = reinterpret_cast<float4*>(st + TG_B_OFF);
                    float4* l4 = reinterpret_cast<float4*>(st + TG_B_OFF + p.BN * 128);
                    const int n4 = p.BN * 8;
                    for (int i0 = ct; i0 < n4; i0 += 4 * TG_ROLE) {
                        float4 v[4];
#pragma unroll
                        for (int l = 0; l < 4; ++l) if (i0 + TG_ROLE * l < n4) v[l] = b4[i0 + TG_ROLE * l];
#pragma unroll
                        for (int l = 0; l < 4; ++l)
                            if (i0 + TG_ROLE * l < n4) {
                                const float4 h = make_float4(tg_rna(v[l].x), tg_rna(v[l].y), tg_rna(v[l].z), tg_rna(v[l].w));
                                b4[i0 + TG_ROLE * l] = h;
                                l4[i0 + TG_ROLE * l] = make_float4(tg_rna(v[l].x - h.x), tg_rna(v[l].y - h.y), tg_rna(v[l].z - h.z), tg_rna(v[l].w - h.w));
                            }
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy stores -> visible to the tensor core
                tg_mbar_arrive(&bar_cvt[s]);
                TG_STAMP(2, 1000 + rit);
            }
        }
    } else {
        // ================= epilogue: TMEM -> registers -> global =================
        const int q = warp & 3, row_l = q * 32 + lane;                 // a warp reads the TMEM lane quadrant (warp % 4)
        const bool dbg_nostore = (g.debug & 1) != 0;
        int tma_seq = 0;
        int seq = 0;
        for (int item = blockIdx.x; item < g.total_items; item += gridDim.x, ++seq) {
            const TGItem it = tg_decode(sp, np, item);
            const TGScalars p = sp[it.pi];      // by value: registers, not re-read after every store / asm
            const int buf = seq % g.n_bufs;
            tg_mbar_wait(&bar_accf[buf], (uint32_t)((seq / g.n_bufs) & 1));
            TG_STAMP(3, seq);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t acc = tmem + (uint32_t)(buf * g.cols_per_buf) + ((uint32_t)(q * 32) << 16);
            const int m = it.m0 + row_l;
            const float bmul = p.bias_mul != 0.f ? p.bias_mul : 1.0f;
            for (int c0 = 0; c0 < p.BN; c0 += 32) {
                __syncwarp();          // lanes leave the previous chunk on different paths; tcgen05.ld is .sync.aligned
                TG_STAMP(3, 4000 + c0);
                float sum[32];
                for (int a = 0; a < p.nmain + (p.merge_corr ? 0 : 1); ++a) {
                    uint32_t v[32];
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                                 : "r"(acc + (uint32_t)(a * p.BN + c0)));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int e = 0; e < 32; ++e) sum[e] = a == 0 ? __uint_as_float(v[e]) : sum[e] + __uint_as_float(v[e]);
                }
                TG_STAMP(3, 2000 + c0);
                if (p.epi == 2) {
                    float* dst = p.partial + ((size_t)it.local * TG_BM + row_l) * p.BN + c0;
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4)
                        asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * g4), "f"(sum[4 * g4]), "f"(sum[4 * g4 + 1]),
                                     "f"(sum[4 * g4 + 2]), "f"(sum[4 * g4 + 3]));
                    continue;
                }
                // The warp's 32 x 32 block is staged in shared memory as [output row][output column] (pitch 36 floats: 128-bit
                // rows, conflict-free both ways) whatever the orientation of the accumulator, and leaves as 128-bit stores: a lane
                // owns 4 consecutive output columns, one store instruction writes 4 output rows x 128 B.  (History, measured with
                // the phase trace: direct lane-per-row stores ~700 cycles per instruction; a generic rolled loop with per-element
                // guards ~3300 cycles per chunk because of ~1000 integer / predicate instructions; this form ~400.)
                float* sw = &epi_stage[warp - 6][0];
                const bool tr = p.transposed != 0;
                if (p.out_tma) {
                    // TMA-store epilogue: bias / ReLU in registers, the warp's 32 x 32 block staged in the 128-byte-swizzled layout
                    // (lane = row writes its eight 16-byte chunks at chunk ^ (row & 7): conflict-free), one cp.async.bulk.tensor
                    // store per block; rows / columns past the matrix are clipped by the tensor map.  Two staging blocks per warp:
                    // the store of chunk i drains while chunk i+1 is read from TMEM.
                    float* blk = &epi_stage[warp - 6][(tma_seq & 1) * 1024];
                    asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");      // the store that last used this block has read it
                    __syncwarp();
                    const float* bp = p.bias ? p.bias + it.n0 + c0 : nullptr;
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4) {
                        float4 v = make_float4(sum[4 * g4], sum[4 * g4 + 1], sum[4 * g4 + 2], sum[4 * g4 + 3]);
                        if (bp) {
                            const int n = it.n0 + c0 + 4 * g4;
                            if (n + 3 < p.Nd) {
                                v.x = fmaf(bmul, __ldg(bp + 4 * g4), v.x); v.y = fmaf(bmul, __ldg(bp + 4 * g4 + 1), v.y);
                                v.z = fmaf(bmul, __ldg(bp + 4 * g4 + 2), v.z); v.w = fmaf(bmul, __ldg(bp + 4 * g4 + 3), v.w);
                            } else {
                                if (n < p.Nd) v.x = fmaf(bmul, __ldg(bp + 4 * g4), v.x);
                                if (n + 1 < p.Nd) v.y = fmaf(bmul, __ldg(bp + 4 * g4 + 1), v.y);
                                if (n + 2 < p.Nd) v.z = fmaf(bmul, __ldg(bp + 4 * g4 + 2), v.z);
                            }
                        }
                        if (p.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        *reinterpret_cast<float4*>(&blk[lane * 32 + 4 * (g4 ^ (lane & 7))]) = v;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0 && !dbg_nostore) {
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                                     ::"l"(&g.p[it.pi].mapOut), "r"(it.n0 + c0), "r"(it.m0 + q * 32), "r"(tg_u32(blk)) : "memory");
                    }
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    ++tma_seq;
                    continue;
                }
                // (warp-uniform condition: every lane of the warp takes the same one of the two paths below)
                const bool direct = !tr && ((p.ldo & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0) && it.n0 + c0 + 32 <= p.Nd &&
                                    (!p.relu_src || (((p.ldrs & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.relu_src) & 15) == 0))) &&
                                    (!p.bias || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0);
                if (direct && m >= p.Md) continue;                      // rows past the matrix
                if (direct) {
                    // rows on the UMMA rows, full aligned chunk: lane = output row, 8 x 128-bit stores straight from registers
                    // (no shared-memory round trip; the 8 stores of a lane complete one 128-byte line)
                    float* dst = p.out + (long long)m * p.ldo + it.n0 + c0;
                    const float* rs = (p.epi == 1 && p.relu_src) ? p.relu_src + (long long)m * p.ldrs + it.n0 + c0 : nullptr;
                    const float* bp = (p.epi == 0 && p.bias) ? p.bias + it.n0 + c0 : nullptr;
                    const bool relu = p.epi == 0 && p.relu, acc = p.accumulate != 0;
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4) {
                        float4 v = make_float4(sum[4 * g4], sum[4 * g4 + 1], sum[4 * g4 + 2], sum[4 * g4 + 3]);
                        if (bp) {
                            float4 b;
                            asm("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(bp + 4 * g4));
                            v.x = fmaf(bmul, b.x, v.x); v.y = fmaf(bmul, b.y, v.y); v.z = fmaf(bmul, b.z, v.z); v.w = fmaf(bmul, b.w, v.w);
                        }
                        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        if (rs) {
                            float4 mk;
                            asm("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(mk.x), "=f"(mk.y), "=f"(mk.z), "=f"(mk.w) : "l"(rs + 4 * g4));
                            if (!(mk.x > 0.f)) v.x = 0.f; if (!(mk.y > 0.f)) v.y = 0.f; if (!(mk.z > 0.f)) v.z = 0.f; if (!(mk.w > 0.f)) v.w = 0.f;
                        }
                        if (acc) {
                            float4 o;
                            asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "l"(dst + 4 * g4));
                            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                        }
                        if (!dbg_nostore)
                            asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * g4), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
                    }
                    continue;
                }
                __syncwarp();
                if (tr) {
#pragma unroll
                    for (int e = 0; e < 32; ++e) sw[e * 36 + lane] = sum[e];           // lane = output column (feature)
                } else {
#pragma unroll
                    for (int g4 = 0; g4 < 8; ++g4)                                       // lane = output row
                        *reinterpret_cast<float4*>(&sw[lane * 36 + 4 * g4]) = make_float4(sum[4 * g4], sum[4 * g4 + 1], sum[4 * g4 + 2], sum[4 * g4 + 3]);
                }
                __syncwarp();
                TG_STAMP(3, 3000 + c0);
                const int orow0 = tr ? it.n0 + c0 : it.m0 + q * 32, ocol0 = tr ? it.m0 + q * 32 : it.n0 + c0;
                const int n_rows = tr ? p.Nd : p.Md, n_cols = tr ? p.Md : p.Nd;
                const int rsub = lane >> 3, col = ocol0 + 4 * (lane & 7);
                const int rows_here = min(32, n_rows - orow0);
                if (rows_here <= 0 || ocol0 >= n_cols) continue;
                const bool vec = ((p.ldo & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0) && ocol0 + 32 <= n_cols &&
                                 (!p.relu_src || (((p.ldrs & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.relu_src) & 15) == 0)));
                if (vec) {
                    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p.epi == 0 && p.bias) {
                        b4.x = bmul * __ldg(p.bias + col); b4.y = bmul * __ldg(p.bias + col + 1);
                        b4.z = bmul * __ldg(p.bias + col + 2); b4.w = bmul * __ldg(p.bias + col + 3);
                    }
                    float* dst = p.out + (long long)(orow0 + rsub) * p.ldo + col;
                    const float* rs = (p.epi == 1 && p.relu_src) ? p.relu_src + (long long)(orow0 + rsub) * p.ldrs + col : nullptr;
                    const long long dstep = 4LL * p.ldo, rstep = 4LL * p.ldrs;
                    const bool relu = p.epi == 0 && p.relu, acc = p.accumulate != 0;
#pragma unroll 4
                    for (int r4 = 0; r4 < 8; ++r4, dst += dstep) {
                        if (4 * r4 + rsub >= rows_here) break;
                        float4 v = *reinterpret_cast<const float4*>(&sw[(4 * r4 + rsub) * 36 + 4 * (lane & 7)]);
                        v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
                        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        if (rs) {
                            float4 m;
                            asm("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(m.x), "=f"(m.y), "=f"(m.z), "=f"(m.w) : "l"(rs + r4 * rstep));
                            if (!(m.x > 0.f)) v.x = 0.f; if (!(m.y > 0.f)) v.y = 0.f; if (!(m.z > 0.f)) v.z = 0.f; if (!(m.w > 0.f)) v.w = 0.f;
                        }
                        if (acc) {
                            float4 o;
                            asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w) : "l"(dst));
                            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                        }
                        if (!dbg_nostore)
                            asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
                    }
                    continue;
                }
                // ragged edge / unaligned output: one element at a time (a lane walks its 4 columns of every 4th row)
#pragma unroll 1
                for (int r4 = 0; r4 < 8; ++r4) {
                    const int r = 4 * r4 + rsub;
                    if (r >= rows_here) break;
#pragma unroll 1
                    for (int e = 0; e < 4; ++e) {
                        const int c = col + e;
                        if (c >= n_cols) break;
                        float v = sw[r * 36 + 4 * (lane & 7) + e];
                        float* dst = p.out + (long long)(orow0 + r) * p.ldo + c;
                        if (p.epi == 0) { if (p.bias) v += bmul * __ldg(p.bias + c); if (p.relu) v = fmaxf(v, 0.f); }
                        else if (p.relu_src && !(tg_ldg_nc(p.relu_src + (long long)(orow0 + r) * p.ldrs + c) > 0.f)) v = 0.f;
                        if (p.accumulate) v += tg_ld_global(dst);
                        if (!dbg_nostore) tg_st_global(dst, v);
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            tg_mbar_arrive(&bar_acce[buf]);
            TG_STAMP(3, 1000 + seq);
        }
    }
    if (warp >= 6) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // the TMA stores have left shared memory and are complete
    if (trace) trace[(warp == 0 ? 0 : warp == 1 ? 1 : warp == 2 ? 2 : 3) * 512 + 510] = tn;
    pdl_trigger();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    __syncwarp();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TG_TMEM_COLS));
}

// Second stage of the split weight gradients: fixed summation order -> bitwise reproducible gradients.
__global__ void __launch_bounds__(256) tgemm_reduce_kernel(const __grid_constant__ TGReduceGroup r) {
    pdl_enter();
    const TGReduceJob& j = r.j[blockIdx.y];
    const int rows = j.K_in + (j.db ? 1 : 0);
    const long long total = (long long)rows * j.N_out;
    const size_t tile = (size_t)TG_BM * j.BN, stride = (size_t)j.n_tiles * j.m_tiles * tile;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int m = (int)(idx / j.N_out), n = (int)(idx % j.N_out);
        const float* src = j.partial + ((size_t)(n / j.BN) * j.m_tiles + m / TG_BM) * tile + (size_t)(m % TG_BM) * j.BN + n % j.BN;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int sp = 0;
        for (; sp + 3 < j.k_splits; sp += 4) {
            s0 += src[(size_t)sp * stride]; s1 += src[(size_t)(sp + 1) * stride];
            s2 += src[(size_t)(sp + 2) * stride]; s3 += src[(size_t)(sp + 3) * stride];
        }
        for (; sp < j.k_splits; ++sp) s0 += src[(size_t)sp * stride];
        const float s = (s0 + s1) + (s2 + s3);
        if (m < j.K_in) j.dw[(long long)n * j.ldw + m] += s;
        else j.db[n] += (j.db_mul != 0.f ? j.db_mul : 1.0f) * s;
    }
}

// ---------------------------------------------------------------- host side ----------------------------------------
namespace {

typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiled encoder() {
    static EncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiled)p;
        cudaGetLastError();
    }
    return fn;
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// 2-D fp32 tensor [outer, inner] with a row pitch in floats; box {32, box_outer}
bool make_map(CUtensorMap* m, const float* base, long long inner, long long outer, long long pitch, int box_outer, bool atom32) {
    EncodeTiled enc = encoder();
    if (!enc || !base || !al16(base) || (pitch & 3) || inner <= 0 || outer <= 0) return false;
    cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    cuuint64_t gstr[1] = {(cuuint64_t)pitch * 4};
    cuuint32_t box[2] = {32, (cuuint32_t)box_outer};
    cuuint32_t est[2] = {1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE,
               atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// N tile: 32-multiples up to `cap`, least padding first, then fewest tiles
int choose_bn(int N, int cap) {
    int best = 32, best_pad = 1 << 30, best_tiles = 1 << 30;
    for (int bn = 32; bn <= cap; bn += 32) {
        const int tiles = cdiv(N, bn), pad = tiles * bn;
        if (pad < best_pad || (pad == best_pad && tiles < best_tiles)) { best = bn; best_pad = pad; best_tiles = tiles; }
    }
    return best;
}

// accumulator plan for a reduction of k8 steps: main accumulators (one per 32 updates, at most 3), and whether the
// correction products may share the single main accumulator (<= 16 steps = 48 updates)
void acc_plan(int k8, int& nmain, int& merge) {
    nmain = k8 > 64 ? 3 : (k8 > 32 ? 2 : 1);
    merge = k8 <= 16 ? 1 : 0;
}
int bn_cap(int nmain, int merge) {
    int cap = (TG_TMEM_COLS / (nmain + (merge ? 0 : 1))) / 32 * 32;
    return cap > 256 ? 256 : cap;
}

float* g_scratch = nullptr;
size_t g_scratch_bytes = 0, g_scratch_cur = 0;

}  // namespace

// Off by default: on the shapes of this path the smem-split 3xTF32 pipeline is bound by shared-memory bandwidth either way
// and the register-staged kernels of linear.cu (several CTAs per SM) are still ahead (profiles/README.md, round 2).
// MARL_B200_TGEMM=1 or marl_tgemm_enable(1) switches every TMA-addressable dense layer over.
static int g_tgemm_on = -1;
bool tgemm_enabled() {
    if (g_tgemm_on < 0) { const char* e = getenv("MARL_B200_TGEMM"); g_tgemm_on = (e && e[0] == '1') ? 1 : 0; }
    return g_tgemm_on == 1 && encoder() != nullptr;
}

float* tgemm_scratch(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (!g_scratch || bytes > g_scratch_bytes) return nullptr;
    if (g_scratch_cur + bytes > g_scratch_bytes) g_scratch_cur = 0;      // ring: regions are consumed by the reduce that follows
    float* p = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(g_scratch) + g_scratch_cur);
    g_scratch_cur += bytes;
    return p;
}

TGBuilder::TGBuilder() : max_bn_(0), max_cols_(0) { memset(&g_, 0, sizeof(g_)); memset(&r_, 0, sizeof(r_)); }

bool TGBuilder::push(TGProblem& P) {
    if (g_.n >= TG_MAXP) return false;
    TGScalars& p = P.s;
    p.item0 = g_.total_items;
    p.n_items = p.m_tiles * p.n_tiles * p.k_splits;
    g_.p[g_.n++] = P;
    g_.total_items += p.n_items;
    if (p.BN > max_bn_) max_bn_ = p.BN;
    const int cols = (p.nmain + (p.merge_corr ? 0 : 1)) * p.BN;
    if (cols > max_cols_) max_cols_ = cols;
    return true;
}

bool TGBuilder::add_fwd(const LinearFwd& a) {
    if (!tgemm_enabled() || g_.n >= TG_MAXP || a.batch != 1 || a.M <= 0 || a.N <= 0) return false;
    const LinOperand& in = a.in;
    const bool plain = in.K2 == 0 && in.onehot_mod == 0;
    const bool agent = in.K1 > 0 && in.K2 > 0 && in.onehot_mod > 0 && !in.onehot_z && in.x_bs == 0 && in.x2_bs == 0 && in.ldx2 == in.K2;
    if (!plain && !agent) return false;
    const int K = lin_width(in);
    if (K > 768 || !al16(a.w) || (a.ldw & 3)) return false;
    TGProblem P;
    memset(&P, 0, sizeof(P));
    TGScalars& p = P.s;
    acc_plan(cdiv(K, TG_BK) * 4, p.nmain, p.merge_corr);
    const int cap = bn_cap(p.nmain, p.merge_corr);
    p.Kd = K;
    p.kb_total = cdiv(K, TG_BK); p.kb_per_split = p.kb_total; p.k_splits = 1;
    p.epi = 0; p.out = a.y; p.ldo = a.ldy; p.accumulate = a.accumulate; p.relu = a.relu; p.bias = a.bias; p.bias_mul = a.bias_mul;
    // every tcgen05.mma costs the same ~190 cycles whatever its N (tools/micro/mma_rate.cu), so narrow layers are computed as
    // y^T = W . x^T: the <= 128 output features sit on the UMMA rows and up to 256 data rows on N -- half the instructions
    p.transposed = (a.N <= TG_BM && a.M >= 256 * 2 * kNumSMs) ? 1 : 0;      // (needs >= 2 waves of 256-row items to pay)
    if (p.transposed) {
        p.BN = cap;
        p.Md = a.N; p.Nd = a.M;
        if (!make_map(&P.mapA, a.w, K, a.N, a.ldw, TG_BM, false)) return false;
        if (!make_map(&P.mapB, in.x, in.K1, a.M, in.ldx, p.BN, false)) return false;
        p.m_tiles = 1; p.n_tiles = cdiv(a.M, p.BN);
    } else {
        p.BN = choose_bn(a.N, cap);
        p.Md = a.M; p.Nd = a.N;
        if (!make_map(&P.mapA, in.x, in.K1, a.M, in.ldx, TG_BM, false)) return false;
        if (!make_map(&P.mapB, a.w, K, a.N, a.ldw, p.BN, false)) return false;
        p.m_tiles = cdiv(a.M, TG_BM); p.n_tiles = cdiv(a.N, p.BN);
    }
    if (!p.transposed && !a.accumulate && al16(a.y) && (a.ldy & 3) == 0) {
        // 32 x 32 output boxes, 128-byte swizzle; the tensor map clips the ragged edges
        EncodeTiled enc = encoder();
        cuuint64_t gdim[2] = {(cuuint64_t)a.N, (cuuint64_t)a.M};
        cuuint64_t gstr[1] = {(cuuint64_t)a.ldy * 4};
        cuuint32_t box[2] = {32, 32}, est[2] = {1, 1};
        if (enc && enc(&P.mapOut, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, a.y, gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
            p.out_tma = 1;
    }
    if (!p.out_tma) P.mapOut = P.mapA;
    if (agent) {
        p.fill_on = p.transposed ? 2 : 1; p.fill_col0 = in.K1; p.fill_A = in.K2; p.fill_N = in.onehot_mod; p.fill_ones = 0;
        p.fill_shift = in.x2_shift; p.fill_period = in.x2_period > 0 ? in.x2_period : 1; p.fill_rows = a.M; p.fill_onehot = in.x2;
    }
    return push(P);
}

bool TGBuilder::add_dgrad(const LinearDgrad& a) {
    if (!tgemm_enabled() || g_.n >= TG_MAXP || a.batch != 1 || a.M <= 0 || a.K <= 0 || a.N <= 0 || a.N > 768) return false;
    TGProblem P;
    memset(&P, 0, sizeof(P));
    TGScalars& p = P.s;
    acc_plan(cdiv(a.N, TG_BK) * 4, p.nmain, p.merge_corr);
    const int cap = bn_cap(p.nmain, p.merge_corr);
    p.Kd = a.N;
    p.kb_total = cdiv(a.N, TG_BK); p.kb_per_split = p.kb_total; p.k_splits = 1;
    p.epi = 1; p.out = a.dx; p.ldo = a.lddx; p.accumulate = a.accumulate; p.relu_src = a.relu_src; p.ldrs = a.ldrs;
    p.transposed = (a.K <= TG_BM && a.M >= 256 * 2 * kNumSMs) ? 1 : 0;
    if (p.transposed) {
        // dx^T = W^T . dy^T: A(m = input feature, k = output unit) = w[k, col0 + m] is MN-major, B = dy is K-major
        p.BN = cap; p.a_mn = 1;
        p.Md = a.K; p.Nd = a.M;
        if (!make_map(&P.mapA, a.w + a.w_col0, a.K, a.N, a.ldw, 32, true)) return false;
        if (!make_map(&P.mapB, a.dy, a.N, a.M, a.lddy, p.BN, false)) return false;
        p.m_tiles = 1; p.n_tiles = cdiv(a.M, p.BN);
    } else {
        p.BN = choose_bn(a.K, cap); p.b_mn = 1;
        p.Md = a.M; p.Nd = a.K;
        if (!make_map(&P.mapA, a.dy, a.N, a.M, a.lddy, TG_BM, false)) return false;
        if (!make_map(&P.mapB, a.w + a.w_col0, a.K, a.N, a.ldw, 32, true)) return false;
        p.m_tiles = cdiv(a.M, TG_BM); p.n_tiles = cdiv(a.K, p.BN);
    }
    return push(P);
}

bool TGBuilder::add_wgrad(const LinearWgrad& a) {
    if (!tgemm_enabled() || g_.n >= TG_MAXP || r_.n >= TG_MAXP || a.batch != 1 || a.M <= 0 || a.N <= 0) return false;
    const LinOperand& in = a.in;
    const bool plain = in.K1 > 0 && in.K2 == 0 && in.onehot_mod == 0;
    const bool shifted = in.K1 == 0 && in.K2 > 0 && in.onehot_mod == 0 && in.x2_bs == 0;               // h_{t-1}
    const bool agent = in.K1 > 0 && in.K2 > 0 && in.onehot_mod > 0 && !in.onehot_z && in.x_bs == 0 && in.x2_bs == 0 && in.ldx2 == in.K2;
    if (!plain && !shifted && !agent) return false;
    const int K_in = lin_width(in);
    const int Md = K_in + (a.db ? 1 : 0);
    TGProblem P;
    memset(&P, 0, sizeof(P));
    TGScalars& p = P.s;
    p.a_mn = 1; p.b_mn = 1;
    p.Md = Md; p.Nd = a.N; p.Kd = a.M;
    // D = in^T . dy  (the transposed weight gradient): M index = input feature, N index = output unit
    if (shifted) {
        if (!make_map(&P.mapA, in.x2, in.K2, a.M, in.ldx2, 32, true)) return false;
        p.a_row_shift = in.x2_shift; p.a_row_period = in.x2_period > 0 ? in.x2_period : 1;
    } else if (!make_map(&P.mapA, in.x, in.K1, a.M, in.ldx, 32, true)) return false;
    const bool dy_tma = al16(a.dy) && (a.lddy & 3) == 0;
    p.BN = choose_bn(a.N, 256);
    if (dy_tma) { if (!make_map(&P.mapB, a.dy, a.N, a.M, a.lddy, 32, true)) return false; }
    else {
        if (a.N > 32 || !a.dy) return false;
        p.BN = 32; p.b_ptr = a.dy; p.ldb = a.lddy; P.mapB = P.mapA;
    }
    if (a.db || agent) {
        p.fill_on = 1;
        p.fill_col0 = agent ? in.K1 : K_in;
        p.fill_A = agent ? in.K2 : 0; p.fill_N = agent ? in.onehot_mod : 0; p.fill_ones = a.db ? 1 : 0;
        p.fill_shift = in.x2_shift; p.fill_period = in.x2_period > 0 ? in.x2_period : 1; p.fill_rows = a.M; p.fill_onehot = in.x2;
    }
    p.m_tiles = cdiv(Md, TG_BM); p.n_tiles = cdiv(a.N, p.BN);
    p.kb_total = cdiv(a.M, TG_BK);
    const int tiles = p.m_tiles * p.n_tiles;
    const int want = kNumSMs / tiles > 0 ? kNumSMs / tiles : 1;      // about one wave of work items per problem
    int kbps = cdiv(p.kb_total, want);
    int kb_max = 24;
    while (kb_max > 8 && (cdiv(kb_max * 4, 32) + 1) * p.BN > TG_TMEM_COLS) kb_max -= 8;     // accumulators must fit in TMEM
    kbps = kbps < 4 ? 4 : (kbps > kb_max ? kb_max : kbps);
    if (kbps > p.kb_total) kbps = p.kb_total;
    p.kb_per_split = kbps; p.k_splits = cdiv(p.kb_total, kbps);
    acc_plan(kbps * 4, p.nmain, p.merge_corr);
    if ((p.nmain + (p.merge_corr ? 0 : 1)) * p.BN > TG_TMEM_COLS) return false;
    p.epi = 2;
    const size_t bytes = (size_t)p.k_splits * tiles * TG_BM * p.BN * sizeof(float);
    p.partial = tgemm_scratch(bytes);
    if (!p.partial) return false;
    if (!push(P)) return false;
    TGReduceJob& j = r_.j[r_.n++];
    j.partial = p.partial; j.k_splits = p.k_splits; j.m_tiles = p.m_tiles; j.n_tiles = p.n_tiles; j.BN = p.BN;
    j.dw = a.dw; j.ldw = a.ldw; j.K_in = K_in; j.N_out = a.N; j.db = a.db; j.db_mul = a.db_mul;
    return true;
}

void TGBuilder::move_reduce_to(TGBuilder& other) {
    for (int i = 0; i < r_.n && other.r_.n < TG_MAXP; ++i) other.r_.j[other.r_.n++] = r_.j[i];
    r_.n = 0;
}

int TGBuilder::launch(cudaStream_t st) {
    if (g_.n == 0) return MARL_OK;
    g_.stage_bytes = TG_B_OFF + 2 * max_bn_ * 128;
    g_.b_off = TG_B_OFF;
    g_.n_stages = TG_RING_BYTES / g_.stage_bytes;
    if (g_.n_stages > TG_MAX_STAGES) g_.n_stages = TG_MAX_STAGES;
    g_.cols_per_buf = max_cols_;
    g_.n_bufs = 2 * max_cols_ <= TG_TMEM_COLS ? 2 : 1;
    { static int dbg = -1; if (dbg < 0) { const char* e = getenv("MARL_TGEMM_DEBUG"); dbg = e ? atoi(e) : 0; } g_.debug = dbg; }
    const size_t smem = 1024 + (size_t)g_.n_stages * g_.stage_bytes;
    static bool attr_done = false;
    if (!attr_done) { cudaFuncSetAttribute(tgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 1024 + TG_RING_BYTES); attr_done = true; }
    const int grid = g_.total_items < kNumSMs ? g_.total_items : kNumSMs;
    {
        if (prof_enabled()) prof_note(g_.p[0].s.Md, g_.p[0].s.Nd, g_.p[0].s.Kd);
        ProfScope ps_("tgemm_kernel", st);
        launch_pdl_prio(linear_prio(), tgemm_kernel, dim3(grid), dim3(TG_THREADS), smem, st, g_);
    }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

int TGBuilder::launch_reduce(cudaStream_t st) {
    if (r_.n == 0) return MARL_OK;
    int max_total = 0;
    for (int i = 0; i < r_.n; ++i) {
        const int t = (r_.j[i].K_in + 1) * r_.j[i].N_out;
        if (t > max_total) max_total = t;
    }
    int bx = cdiv(max_total, 256);
    if (bx > 64) bx = 64;
    {
        ProfScope ps_("tgemm_reduce_kernel", st);
        launch_pdl_prio(linear_prio(), tgemm_reduce_kernel, dim3(bx, r_.n), dim3(256), 0, st, r_);
    }
    MARL_LAUNCH_CHECK();
    r_.n = 0;
    return MARL_OK;
}

}  // namespace marl

// Debug: phase trace of CTA 0 of the tgemm launches that follow (on = 1 allocates / clears the buffer); dump copies the
// 4 x 512 (tag, clock64) words to the host.
extern "C" int marl_tgemm_trace(int on, long long* host_out /* 2048 or null */) {
    static long long* buf = nullptr;
    if (on && !buf) { if (cudaMalloc(&buf, 2048 * sizeof(long long)) != cudaSuccess) return MARL_EINVAL; }
    if (on && buf) cudaMemset(buf, 0, 2048 * sizeof(long long));
    if (host_out && buf) { cudaDeviceSynchronize(); cudaMemcpy(host_out, buf, 2048 * sizeof(long long), cudaMemcpyDeviceToHost); }
    long long* v = on ? buf : nullptr;
    marl::g_trace_host = v;
    cudaMemcpyToSymbol(marl::g_tg_trace, &v, sizeof(v));
    return MARL_OK;
}

extern "C" int marl_tgemm_enable(int on) {
    const int prev = marl::tgemm_enabled() ? 1 : 0;
    marl::g_tgemm_on = on ? 1 : 0;
    return prev;
}

extern "C" int marl_set_deterministic(int on) {
    const int prev = marl::deterministic_wgrad() ? 1 : 0;
    marl::set_deterministic_wgrad(on);
    return prev;
}

extern "C" int marl_set_scratch(void* ptr, size_t bytes) {
    marl::g_scratch = reinterpret_cast<float*>(ptr);
    marl::g_scratch_bytes = ptr ? bytes : 0;
    marl::g_scratch_cur = 0;
    return MARL_OK;
}

// Test / bench hooks for the dense primitives (plain row-major operands):
//   fwd  : y[M,N]   = act(x[M,K] . w[N,K]^T + bias)
//   dgrad: dx[M,K]  = (dy[M,N] . w[N,K]) * (relu_src > 0)
//   wgrad: dw[N,K] += dy[M,N]^T . x[M,K] ; db[N] += colsum(dy)
extern "C" int marl_linear_fwd(const float* x, int ldx, const float* w, int ldw, const float* bias, float* y, int ldy,
                               int M, int N, int K, int relu, void* stream) {
    if (!x || !w || !y || M <= 0 || N <= 0 || K <= 0) return MARL_EINVAL;
    marl::LinearFwd f{};
    f.in = marl::plain_operand(x, ldx, K); f.w = w; f.ldw = ldw; f.bias = bias; f.y = y; f.ldy = ldy; f.M = M; f.N = N; f.relu = relu; f.batch = 1;
    return marl::linear_fwd(f, (cudaStream_t)stream);
}
extern "C" int marl_linear_dgrad(const float* dy, int lddy, const float* w, int ldw, const float* relu_src, int ldrs, float* dx,
                                 int lddx, int M, int N, int K, void* stream) {
    if (!dy || !w || !dx || M <= 0 || N <= 0 || K <= 0) return MARL_EINVAL;
    marl::LinearDgrad g{};
    g.dy = dy; g.lddy = lddy; g.w = w; g.ldw = ldw; g.dx = dx; g.lddx = lddx; g.relu_src = relu_src; g.ldrs = ldrs;
    g.M = M; g.N = N; g.K = K; g.batch = 1;
    return marl::linear_dgrad(g, (cudaStream_t)stream);
}
extern "C" int marl_linear_wgrad(const float* dy, int lddy, const float* x, int ldx, float* dw, int ldw, float* db, int M, int N,
                                 int K, void* stream) {
    if (!dy || !x || !dw || M <= 0 || N <= 0 || K <= 0) return MARL_EINVAL;
    marl::LinearWgrad w{};
    w.dy = dy; w.lddy = lddy; w.in = marl::plain_operand(x, ldx, K); w.dw = dw; w.ldw = ldw; w.db = db; w.M = M; w.N = N; w.batch = 1;
    return marl::linear_wgrad(w, (cudaStream_t)stream);
}
