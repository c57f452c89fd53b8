// Dense-layer primitives: forward, data-gradient and weight-gradient GEMMs on the 5th-generation tensor
// cores.  One CTA owns a 128 x 64 output tile: operands are staged in shared memory in the canonical
// K-major (no-swizzle) UMMA layout, a single elected thread issues tcgen05.mma kind::tf32 (M=128, N=64,
// K=8) with the accumulator in tensor memory (TMEM), completion is tracked with tcgen05.commit ->
// mbarrier, and the epilogue reads the accumulator back with tcgen05.ld.
//
// Accuracy: the parity gate on losses / gradients is 1e-5 relative, which a single TF32 pass (2^-11)
// cannot meet.  Every operand tile is therefore stored twice, x = hi + lo with hi = rna_tf32(x) and
// lo = rna_tf32(x - hi), and each k-step issues
//     D += A_lo.B_hi ;  D += A_hi.B_lo ;  D += A_hi.B_hi            (3xTF32, ~5e-7 relative, fp32 accumulate)
// -- measured with tools/micro/tc5_probe.cu.
//
// They replace the cuBLAS addmm calls behind nn.Linear in the reference (network/q_network.py:17,20;
// network/mixer.py:45-55,117-145,200-206,365-375,399-409) and their autograd duals.
#include "linear.h"
#include "umma.cuh"
#include "tgemm.h"
#include "profile.h"

namespace marl {

constexpr int UM = 128, UN = 64, UK = 16, UT = 256;   // CTA tile (UMMA M, N), k-tile, producer / epilogue threads
constexpr int UTH = UT + 32;                          // + one warp whose lane 0 issues the MMAs
constexpr int kKChunks = UK / 4;                       // 16-byte k-chunks per k-tile
// Canonical K-major layout: element (row, k) at float offset (k/4)*PITCH + row*4 + k%4, i.e. 8 rows x 16 B
// core matrices, SBO = 128 B between 8-row groups, LBO = PITCH*4 B between k-chunks.  PITCH = ROWS*4 + 8
// keeps both the 128-bit stores of k-contiguous operands and the scalar stores of transposed operands
// (almost) free of bank conflicts.
constexpr int A_PITCH = UM * 4 + 8, B_PITCH = UN * 4 + 8;
// MN-major layout for operands whose memory is contiguous along the OUTPUT index (both operands of a weight gradient, W of a
// data gradient).  For 32-bit operands the tensor core knows exactly one: SWIZZLE_128B_BASE32B (cutlass sm100_common.inl: "for
// mn-major tf32 operands, SW128_32B is the only available smem layout"; validated with TMA-written tiles in tools/micro/
// tma_probe.cu).  A "box" is 32 output indices wide: per reduction index k one 128-byte row of 32 consecutive output elements;
// atoms of 4 k-rows (512 B, SBO), two atoms per K = 8 step, boxes LBO apart; inside a row the four 32-byte chunks are XORed with
// (k & 3).  A quad of 4 consecutive output indices at one k is ONE 128-bit store -- no transposing scalar stores.
#ifndef MARL_MN_MAJOR
#define MARL_MN_MAJOR 1
#endif
constexpr bool kMnMajor = MARL_MN_MAJOR != 0;
constexpr int MN_BOX_BYTES = UK * 128;                                // one box of a k-tile: UK rows x 128 B
// >= the K-major (8320 / 4224 B) and MN-major (8192 / 4096 B) tiles, multiples of 512 B (the swizzle atom); two stages + alignment
// slack stay under 56 KB so that four CTAs share an SM (at 57 KB -- three CTAs -- the step was 20 us slower)
constexpr int kAFloats = kMnMajor ? 8704 / 4 : kKChunks * A_PITCH, kBFloats = kMnMajor ? 4608 / 4 : kKChunks * B_PITCH;
static_assert(!kMnMajor || (kAFloats * 4 >= (UM / 32) * MN_BOX_BYTES && kBFloats * 4 >= (UN / 32) * MN_BOX_BYTES), "MN-major tile");
static_assert(kAFloats >= kKChunks * A_PITCH && kBFloats >= kKChunks * B_PITCH, "K-major tile");

struct alignas(kMnMajor ? 1024 : 128) UmmaStage {
    float a_hi[kAFloats];
    float a_lo[kAFloats];
    float b_hi[kBFloats];
    float b_lo[kBFloats];
};
constexpr int kUmmaStages = 2;
// k-tiles a producer thread keeps in flight in registers.  Measured 2 / 3 / 4 / 6 deep (gpurun_out/ab_fd.txt): no gain
// stand-alone (9.4 / 9.6 / 9.9 / 14.4 us for 19200 x 64 x 96) -- 4 costs 96 registers (2 CTAs per SM instead of 3), 6 is slower.
#ifndef MARL_FETCH_DEPTH
#define MARL_FETCH_DEPTH 2
#endif
constexpr int kFetchDepth = MARL_FETCH_DEPTH;
// Accumulators per CTA tile in TMEM.  The tensor core adds every K=8 product block into the fp32 accumulator
// with truncation, an error that grows with the NUMBER of accumulator updates; the hi.hi products are
// therefore dealt round-robin to kAccMain accumulators, the two (2^-11 smaller) correction products go to
// their own accumulator, and the epilogue adds the four up in fp32.
constexpr int kAccMain = 3, kAccAll = kAccMain + 1, kTmemCols = 256;
static_assert(kAccAll * UN <= kTmemCols, "TMEM allocation too small");
// short reductions (<= 32 accumulator updates) keep one main accumulator: reading TMEM back costs ~0.25 us each
__host__ __device__ __forceinline__ int acc_main_count(int nsteps) { return nsteps > 32 ? kAccMain : 1; }
constexpr size_t kUmmaSmem = kUmmaStages * sizeof(UmmaStage) + (kMnMajor ? 1024 : 128);

// 32-bit instruction descriptor: D = F32, A = B = TF32, both K-major, N >> 3 at bit 17, M >> 4 at bit 24.
constexpr uint32_t kUmmaIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(UN >> 3) << 17) | ((uint32_t)(UM >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate, uint32_t idesc = kUmmaIdesc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Per-thread share of one k-tile and where it lands in shared memory.
//   RED operand (memory contiguous along the reduction): quad = 4 consecutive reduction elements of one
//     row -> one 128-bit store;
//   otherwise (contiguous along the output index): quad = rows i..i+3 at one reduction index, fetched with
//     the 16 reduction indices of the tile across neighbouring lanes -> 4 scalar stores (the transpose into
//     the K-major layout the tensor core wants for 32-bit operands).
template <bool RED, int ROWS, int NQ>
struct QuadMap {
    int i[NQ], r[NQ];
    int off[NQ];             // where the quad lands in a stage array (floats), fixed for the whole loop
    __device__ __forceinline__ QuadMap(int pitch = ROWS * 4 + 8) {
#pragma unroll
        for (int l = 0; l < NQ; ++l) {
            const int q = threadIdx.x + l * UT;
            if (RED) { i[l] = q >> 2; r[l] = (q & 3) * 4; }
            else if (kMnMajor) {      // a warp = 8 quads (one 128-byte box row) x 4 reduction indices: coalesced loads, conflict-free stores
                const int u = q & 7, kr4 = (q >> 3) & 3, box = (q >> 5) % (ROWS / 32), kg = q / (ROWS);
                i[l] = (box * 8 + u) * 4; r[l] = kg * 4 + kr4;
            }
            else { i[l] = (q >> 4) * 4; r[l] = q & 15; }
            if (RED) off[l] = (r[l] >> 2) * pitch + i[l] * 4;
            else if (kMnMajor) {
                const int u = (i[l] >> 2) & 7, box = i[l] >> 5;        // 16-byte unit inside the box row, box
                off[l] = (box * MN_BOX_BYTES + (r[l] >> 2) * 512 + (r[l] & 3) * 128 + ((((u >> 1) ^ (r[l] & 3)) << 5) | ((u & 1) << 4))) >> 2;
            } else off[l] = (r[l] >> 2) * pitch + i[l] * 4 + (r[l] & 3);
        }
    }
    static __device__ __forceinline__ void store(float* hi, float* lo, int off, const float4& v) {
        float4 h, l;
        tf32_split(v.x, h.x, l.x); tf32_split(v.y, h.y, l.y); tf32_split(v.z, h.z, l.z); tf32_split(v.w, h.w, l.w);
        if (RED || kMnMajor) {
            *reinterpret_cast<float4*>(hi + off) = h;
            *reinterpret_cast<float4*>(lo + off) = l;
        } else {
            hi[off] = h.x; hi[off + 4] = h.y; hi[off + 8] = h.z; hi[off + 12] = h.w;
            lo[off] = l.x; lo[off + 4] = l.y; lo[off + 8] = l.z; lo[off + 12] = l.w;
        }
    }
};

struct UmmaCtx {
    UmmaStage* stages;
    uint64_t* bars;        // [kUmmaStages] "MMAs that read this stage are done"
    uint32_t tmem;         // TMEM base (lane 0, first of UN columns)
};

// CTA prologue: carve shared memory, init the mbarriers, allocate UN TMEM columns (warp 0).
__device__ __forceinline__ uint32_t tmem_cols_for(int nsteps) { return acc_main_count(nsteps) > 1 ? (uint32_t)kTmemCols : 2u * UN; }

__device__ __forceinline__ UmmaCtx umma_setup(unsigned char* smem_raw, int nsteps) {
    __shared__ uint64_t bars[kUmmaStages];
    __shared__ uint32_t tmem_base;
    UmmaCtx c;
    constexpr uintptr_t kAlign = kMnMajor ? 1023 : 127;
    c.stages = reinterpret_cast<UmmaStage*>((reinterpret_cast<uintptr_t>(smem_raw) + kAlign) & ~kAlign);
    c.bars = bars;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kUmmaStages; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bars[s])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(tmem_cols_for(nsteps)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    c.tmem = tmem_base;
    return c;
}

__device__ __forceinline__ void umma_teardown(const UmmaCtx& c, int nsteps) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(c.tmem), "r"(tmem_cols_for(nsteps)));
}

// Main loop over the reduction range [rbeg, rend): global -> registers (two k-tiles ahead) -> shared (hi, lo)
// -> tcgen05.mma.  FA(i, r) / FB(j, r) return the operand quad as a float4.  BIAS (weight gradient only)
// also accumulates the column sums of the A operand into bsum.
template <bool A_RED, bool B_RED, int BIAS, class OA, class OB>      // BIAS: 0 none, 1 column sums of the A operand, 2 of the B operand
__device__ __forceinline__ void umma_loop(const UmmaCtx& c, const OA& A, const OB& B, int i0, int j0, int rbeg, int rend, float (&bsum)[2][4]) {
    const QuadMap<A_RED, UM, 2> ma;
    const QuadMap<B_RED, UN, 1> mb;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int nk = (rend - rbeg + UK - 1) / UK;
    const int nmain = acc_main_count(nk * (UK / 8));
    float4 ra[kFetchDepth][2], rb[kFetchDepth];   // register sets: tiles kt .. kt+kFetchDepth-1 in flight
    // RED operands (operand row = tile row, contiguous along the reduction): row context hoisted out of the loop;
    // otherwise the operand row IS the reduction index and changes with every tile
    typename OA::Row arow[2]; typename OB::Row brow;
    if (threadIdx.x < UT) {
        if (A_RED) { arow[0] = A.row(i0 + ma.i[0]); arow[1] = A.row(i0 + ma.i[1]); }
        if (B_RED) brow = B.row(j0 + mb.i[0]);
    }
    auto fetch = [&](int kt, int set) {
        const int r0 = rbeg + kt * UK;
#pragma unroll
        for (int l = 0; l < 2; ++l) {
            const int r = r0 + ma.r[l];
            ra[set][l] = (kt < nk && r < rend) ? (A_RED ? A.quad_at(arow[l], r) : A.quad(r, i0 + ma.i[l])) : zero4;
        }
        const int r = r0 + mb.r[0];
        rb[set] = (kt < nk && r < rend) ? (B_RED ? B.quad_at(brow, r) : B.quad(r, j0 + mb.i[0])) : zero4;
    };
    if (threadIdx.x >= UT) {
        // ---- MMA warp.  A clock64 trace of the single-role version showed the issuing thread busy for 700-900 cycles
        // per k-tile (six tcgen05.mma + descriptors) while the other 255 threads waited for it at the next barrier;
        // here the producers only ARRIVE on a named barrier and go on fetching, this warp SYNCs on it and issues.
        for (int kt = 0; kt < nk; ++kt) {
            const int s = kt & 1;
            asm volatile("bar.sync %0, %1;" ::"r"(1 + s), "n"(UTH) : "memory");      // stage s written and proxy-fenced by all producers
            if (threadIdx.x == UT) {
                UmmaStage& st = c.stages[s];
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                constexpr bool A_MN = !A_RED && kMnMajor, B_MN = !B_RED && kMnMajor;
                constexpr uint32_t idesc = kUmmaIdesc | (A_MN ? (1u << 15) : 0u) | (B_MN ? (1u << 16) : 0u);
                for (int k8 = 0; k8 < UK / 8; ++k8) {
                    // K-major: two 16-byte k-chunks per step, LBO = chunk pitch, SBO = 128 B between 8-row groups
                    // MN-major: two 4-row atoms (1 KB) per step, LBO = box pitch, SBO = 512 B between atoms
                    const uint32_t ao = A_MN ? (uint32_t)k8 * 1024u : (uint32_t)(2 * k8) * A_PITCH * 4;
                    const uint32_t bo = B_MN ? (uint32_t)k8 * 1024u : (uint32_t)(2 * k8) * B_PITCH * 4;
                    const uint32_t albo = A_MN ? MN_BOX_BYTES : A_PITCH * 4, asbo = A_MN ? 512 : 128;
                    const uint32_t blbo = B_MN ? MN_BOX_BYTES : B_PITCH * 4, bsbo = B_MN ? 512 : 128;
                    const uint64_t amn = A_MN ? ((uint64_t)1 << 61) : 0, bmn = B_MN ? ((uint64_t)1 << 61) : 0;   // layout type 1 = SWIZZLE_128B_BASE32B
                    const uint64_t dah = umma_desc(smem_u32(st.a_hi) + ao, albo, asbo) | amn, dal = umma_desc(smem_u32(st.a_lo) + ao, albo, asbo) | amn;
                    const uint64_t dbh = umma_desc(smem_u32(st.b_hi) + bo, blbo, bsbo) | bmn, dbl = umma_desc(smem_u32(st.b_lo) + bo, blbo, bsbo) | bmn;
                    const int step = kt * (UK / 8) + k8;                       // global k8 index of this CTA
                    umma_tf32(c.tmem + nmain * UN, dal, dbh, step ? 1u : 0u, idesc);      // corrections
                    umma_tf32(c.tmem + nmain * UN, dah, dbl, 1u, idesc);
                    umma_tf32(c.tmem + (step % nmain) * UN, dah, dbh, step >= nmain ? 1u : 0u, idesc);
                }
                umma_commit(&c.bars[s]);
            }
            __syncwarp();
        }
        return;
    }
#pragma unroll
    for (int d = 0; d < kFetchDepth; ++d) fetch(d, d);
    for (int kt0 = 0; kt0 < nk; kt0 += kFetchDepth) {
#pragma unroll
        for (int d = 0; d < kFetchDepth; ++d) {          // (unrolled: the register set index must be static)
            const int kt = kt0 + d;
            if (kt >= nk) break;
            const int s = kt & 1;
            UmmaStage& st = c.stages[s];
            if (kt >= kUmmaStages) mbar_wait(&c.bars[s], (uint32_t)((kt / kUmmaStages - 1) & 1));   // MMAs of tile kt-2 have read this stage
#pragma unroll
            for (int l = 0; l < 2; ++l) {
                const float4 v = ra[d][l];
                QuadMap<A_RED, UM, 2>::store(st.a_hi, st.a_lo, ma.off[l], v);
                if (BIAS == 1) { bsum[l][0] += v.x; bsum[l][1] += v.y; bsum[l][2] += v.z; bsum[l][3] += v.w; }
            }
            QuadMap<B_RED, UN, 1>::store(st.b_hi, st.b_lo, mb.off[0], rb[d]);
            if (BIAS == 2) { bsum[0][0] += rb[d].x; bsum[0][1] += rb[d].y; bsum[0][2] += rb[d].z; bsum[0][3] += rb[d].w; }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy stores -> visible to the tensor core
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            asm volatile("bar.arrive %0, %1;" ::"r"(1 + s), "n"(UTH) : "memory");   // hand the stage to the MMA warp, do not wait for it
            fetch(kt + kFetchDepth, d);                   // refill the register set just consumed
        }
    }
    // all MMAs done: the last commit of each stage covers everything issued before it
    const int last = nk - 1;
    if (nk >= 1) mbar_wait(&c.bars[last & 1], (uint32_t)((last / kUmmaStages) & 1));
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// Epilogue: warp w reads TMEM lanes 32*(w%4).. (= tile rows) and 32 of the 64 columns ((w/4)*32..);
// f(row_in_tile, col_in_tile, v[4]) is called for each group of 4 consecutive columns.
template <class F>
__device__ __forceinline__ void umma_epilogue(const UmmaCtx& c, int nsteps, F f) {
    if (threadIdx.x >= UT) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = (warp & 3) * 32 + lane, c0 = (warp >> 2) * 32;
    const int nmain = acc_main_count(nsteps);
    float sum[32];
#pragma unroll
    for (int acc = 0; acc < kAccAll; ++acc) {
        if (acc > nmain) continue;                            // main accumulators 0..nmain-1, corrections at nmain
        uint32_t v[32];
        const uint32_t taddr = c.tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(acc * UN + c0);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                       "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                       "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                       "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                     : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int e = 0; e < 32; ++e) sum[e] = (acc == 0) ? __uint_as_float(v[e]) : sum[e] + __uint_as_float(v[e]);
    }
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        float o[4] = {sum[4 * g], sum[4 * g + 1], sum[4 * g + 2], sum[4 * g + 3]};
        f(row, c0 + 4 * g, o);
    }
}

// y[M,N] (+)= act(in . w^T + bias)
template <bool VEC_A, bool VEC_B>
__global__ void __launch_bounds__(UTH) linear_fwd_kernel(LinearFwd a) {
    extern __shared__ unsigned char umma_smem[];
    const int K = lin_width(a.in);
    const int nsteps = ((K + UK - 1) / UK) * (UK / 8);
    const UmmaCtx c = umma_setup(umma_smem, nsteps);       // barriers + TMEM: no global memory, overlaps the predecessor's tail
    pdl_wait();
    const int z = blockIdx.z, m0 = blockIdx.x * UM, n0 = blockIdx.y * UN;
    const OpLin A{a.in, z, a.M, K, VEC_A, VEC_A && vec2_ok(a.in)};               // rows m, reduction k (contiguous)
    const OpMat B{a.w + (long long)z * a.w_bs, a.ldw, a.N, K, VEC_B};             // rows n, reduction k (contiguous)
    float unused[2][4];
    umma_loop<true, true, 0>(c, A, B, m0, n0, 0, K, unused);
    pdl_trigger();                       // main loop done: the next kernel's CTAs may take the freed slots
    const float* bias = a.bias ? a.bias + (long long)z * a.b_bs : nullptr;
    float* y = a.y + (long long)z * a.y_bs;
    const float bmul = a.bias_mul != 0.f ? a.bias_mul : 1.0f;
    const bool vec_out = ((a.ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(y) & 15) == 0) && !a.accumulate;
    __shared__ float sbias[UN];          // the tile's bias slice, fetched once per CTA
    if (threadIdx.x < UN) sbias[threadIdx.x] = (bias && n0 + threadIdx.x < a.N) ? bmul * __ldg(bias + n0 + threadIdx.x) : 0.f;
    __syncthreads();
    umma_epilogue(c, nsteps, [&](int i, int j, float (&v)[4]) {
        const int m = m0 + i, n = n0 + j;
        if (m >= a.M || n >= a.N) return;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            v[e] += sbias[j + e];
            if (a.relu) v[e] = fmaxf(v[e], 0.f);
        }
        float* dst = y + (long long)m * a.ldy + n;
        if (vec_out && n + 3 < a.N) { *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]); return; }
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (n + e < a.N) dst[e] = a.accumulate ? dst[e] + v[e] : v[e];
    });
    umma_teardown(c, nsteps);
}

// dx[M,K] (+)= (dy[M,N] . w[N, col0:col0+K]) * (relu_src > 0)
template <bool VEC_A, bool VEC_B, bool WT = false>
__global__ void __launch_bounds__(UTH) linear_dgrad_kernel(LinearDgrad a) {
    extern __shared__ unsigned char umma_smem[];
    const int nsteps = ((a.N + UK - 1) / UK) * (UK / 8);
    const UmmaCtx c = umma_setup(umma_smem, nsteps);       // barriers + TMEM: no global memory, overlaps the predecessor's tail
    pdl_wait();
    const int z = blockIdx.z, m0 = blockIdx.x * UM, k0 = blockIdx.y * UN;
    const OpMat A{a.dy + (long long)z * a.dy_bs, a.lddy, a.M, a.N, VEC_A};               // rows m, reduction n (contiguous)
    float unused[2][4];
    if (WT) {
        const OpMat Bt{a.wt, a.ldwt, a.K, a.N, true};                                    // rows k, reduction n (contiguous): pre-transposed
        umma_loop<true, true, 0>(c, A, Bt, m0, k0, 0, a.N, unused);
    } else {
        const OpMat B{a.w + (long long)z * a.w_bs + a.w_col0, a.ldw, a.N, a.K, VEC_B};   // rows n (reduction), cols k (contiguous)
        umma_loop<true, false, 0>(c, A, B, m0, k0, 0, a.N, unused);
    }
    pdl_trigger();                       // main loop done: the next kernel's CTAs may take the freed slots
    float* dx = a.dx + (long long)z * a.dx_bs;
    const float* rs = a.relu_src ? a.relu_src + (long long)z * a.rs_bs : nullptr;
    const bool vec_rs = rs && ((a.ldrs & 3) == 0) && ((reinterpret_cast<uintptr_t>(rs) & 15) == 0);
    const bool vec_dx = ((a.lddx & 3) == 0) && ((reinterpret_cast<uintptr_t>(dx) & 15) == 0);
    umma_epilogue(c, nsteps, [&](int i, int j, float (&v)[4]) {
        const int m = m0 + i, k = k0 + j;
        if (m >= a.M || k >= a.K) return;
        const bool full = k + 3 < a.K;
        if (rs) {
            float r4[4] = {1.f, 1.f, 1.f, 1.f};
            if (vec_rs && full) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(rs + (long long)m * a.ldrs + k));
                r4[0] = t.x; r4[1] = t.y; r4[2] = t.z; r4[3] = t.w;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (k + e < a.K) r4[e] = __ldg(rs + (long long)m * a.ldrs + k + e);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) if (!(r4[e] > 0.0f)) v[e] = 0.0f;
        }
        float* dst = dx + (long long)m * a.lddx + k;
        if (vec_dx && full) {
            float4 o = make_float4(v[0], v[1], v[2], v[3]);
            if (a.accumulate) { const float4 t = *reinterpret_cast<float4*>(dst); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
            *reinterpret_cast<float4*>(dst) = o;
            return;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) if (k + e < a.K) dst[e] = a.accumulate ? dst[e] + v[e] : v[e];
    });
    umma_teardown(c, nsteps);
}

// dw[N, 0:K] += dy^T . in ; db[N] += colsum(dy).  Split over the M rows (blockIdx.z).  With a scratch arena (`part`) every
// split stores its tile to part[blockIdx.z][N][ldp] and wgrad_reduce_kernel adds the splits in a fixed order (bitwise
// reproducible gradients); without one the splits meet in atomics on the output.
template <bool VEC_A, bool VEC_B>
__global__ void __launch_bounds__(UTH, 3) linear_wgrad_kernel(LinearWgrad a, int splits, int chunk, float* part, float* part_b, int ldp) {
    extern __shared__ unsigned char umma_smem[];
    const int zb = blockIdx.z / splits, sp = blockIdx.z % splits;
    const int i0 = blockIdx.x * UM, j0 = blockIdx.y * UN;
    const int K = lin_width(a.in);
    const int mbeg = sp * chunk, mend = min(a.M, mbeg + chunk);
    const int nsteps = mend > mbeg ? ((mend - mbeg + UK - 1) / UK) * (UK / 8) : 0;
    const UmmaCtx c = umma_setup(umma_smem, nsteps);       // barriers + TMEM: no global memory, overlaps the predecessor's tail
    pdl_wait();
    const OpMat A{a.dy + (long long)zb * a.dy_bs, a.lddy, a.M, a.N, VEC_A};      // rows m (reduction), cols n
    const OpLin B{a.in, zb, a.M, K, VEC_B, VEC_B && vec2_ok(a.in)};             // rows m (reduction), cols k
    float bsum[2][4] = {};
    const bool want_bias = a.db != nullptr && blockIdx.y == 0;
    if (want_bias) umma_loop<false, false, 1>(c, A, B, i0, j0, mbeg, mend, bsum);
    else umma_loop<false, false, 0>(c, A, B, i0, j0, mbeg, mend, bsum);
    pdl_trigger();                       // main loop done: the next kernel's CTAs may take the freed slots
    if (kMnMajor) {
        // the quads of one 4-wide output group are spread over 8 threads (two reduction indices each): fold them through shared
        // memory, the first 128 threads publish
        // (the stage ring is free again: umma_loop returns when every MMA has read it.  A static array here would push the CTA
        // past 56 KB and cost the fourth CTA per SM)
        float (*sb)[UM] = reinterpret_cast<float (*)[UM]>(c.stages);
        if (want_bias && threadIdx.x < UT) {
            const QuadMap<false, UM, 2> ma;                            // both quads of a thread sit on the same output group
            const int slot = ((threadIdx.x >> 3) & 3) + 4 * (threadIdx.x >> 7);      // (reduction index mod 4, k-group): 8 threads per group
#pragma unroll
            for (int e = 0; e < 4; ++e) sb[slot][ma.i[0] + e] = bsum[0][e] + bsum[1][e];
        }
        __syncthreads();
        if (want_bias && threadIdx.x < UM) {
            const float bmul = a.db_mul != 0.f ? a.db_mul : 1.0f;
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < UT / 32; ++w) v += sb[w][threadIdx.x];
            const int n = i0 + threadIdx.x;
            if (n < a.N) {
                if (part_b) part_b[(long long)blockIdx.z * a.N + n] = bmul * v;
                else atomicAdd(a.db + (long long)zb * a.db_bs + n, bmul * v);
            }
        }
    } else if (want_bias && threadIdx.x < UT) {
        // the 16 reduction indices of a k-tile sit in 16 neighbouring lanes: fold them, lane r == 0 publishes
        const QuadMap<false, UM, 2> ma;
        const float bmul = a.db_mul != 0.f ? a.db_mul : 1.0f;
#pragma unroll
        for (int l = 0; l < 2; ++l)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float v = bsum[l][e];
                v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2);
                v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 8);
                const int n = i0 + ma.i[l] + e;
                if (ma.r[l] == 0 && n < a.N) {
                    if (part_b) part_b[(long long)blockIdx.z * a.N + n] = bmul * v;
                    else atomicAdd(a.db + (long long)zb * a.db_bs + n, bmul * v);
                }
            }
    }
    float* dw = a.dw + (long long)zb * a.dw_bs;
    if (part && mbeg >= mend) {      // (cannot happen with the host's split plan; keeps the reduce well-defined)
        for (int idx = threadIdx.x; idx < UM * UN; idx += UTH) {
            const int n = i0 + idx / UN, k = j0 + idx % UN;
            if (n < a.N && k < K) part[((long long)blockIdx.z * a.N + n) * ldp + k] = 0.f;
        }
    }
    const bool vec_dw = ((a.ldw & 3) == 0) && ((reinterpret_cast<uintptr_t>(dw) & 15) == 0);
    if (mbeg < mend)
        umma_epilogue(c, nsteps, [&](int i, int j, float (&v)[4]) {
            const int n = i0 + i, k = j0 + j;
            if (n >= a.N || k >= K) return;
            if (part) {      // ldp is a multiple of 4 and the arena is 256-byte aligned: one 128-bit store
                float* pd = part + ((long long)blockIdx.z * a.N + n) * ldp + k;
                if (k + 3 < ldp) { *reinterpret_cast<float4*>(pd) = make_float4(v[0], v[1], v[2], v[3]); return; }
#pragma unroll
                for (int e = 0; e < 4; ++e) if (k + e < K) pd[e] = v[e];
                return;
            }
            float* dst = dw + (long long)n * a.ldw + k;
            if (vec_dw && k + 3 < K) {      // one 128-bit reduction instead of four atomics
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
                return;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (k + e < K) atomicAdd(dst + e, v[e]);
        });
    umma_teardown(c, nsteps);
}

// The same product with the roles of the operands swapped: the tile's 128 rows walk the INPUT width k, its 64 columns the
// outputs n (acc[k][n] = sum_m in[m][k] dy[m][n], stored transposed).  Fewer tiles whenever N <= 64 < K (fc1 of the agent:
// 64 x 96 -> one tile instead of two, 64 x 150 -> two instead of three, 64 x 348 -> three instead of six), each with a full A
// operand instead of a half-empty one; the column sums of dy (db) come from the B operand of the k-tile 0 CTAs.
template <bool VEC_A, bool VEC_B>
__global__ void __launch_bounds__(UTH, 3) linear_wgrad_swap_kernel(LinearWgrad a, int splits, int chunk, float* part, float* part_b, int ldp) {
    extern __shared__ unsigned char umma_smem[];
    const int zb = blockIdx.z / splits, sp = blockIdx.z % splits;
    const int k0 = blockIdx.x * UM, n0 = blockIdx.y * UN;
    const int K = lin_width(a.in);
    const int mbeg = sp * chunk, mend = min(a.M, mbeg + chunk);
    const int nsteps = mend > mbeg ? ((mend - mbeg + UK - 1) / UK) * (UK / 8) : 0;
    const UmmaCtx c = umma_setup(umma_smem, nsteps);
    pdl_wait();
    const OpLin A{a.in, zb, a.M, K, VEC_B, VEC_B && vec2_ok(a.in)};             // rows m (reduction), cols k
    const OpMat B{a.dy + (long long)zb * a.dy_bs, a.lddy, a.M, a.N, VEC_A};      // rows m (reduction), cols n
    float bsum[2][4] = {};
    const bool want_bias = a.db != nullptr && blockIdx.x == 0;
    if (want_bias) umma_loop<false, false, 2>(c, A, B, k0, n0, mbeg, mend, bsum);
    else umma_loop<false, false, 0>(c, A, B, k0, n0, mbeg, mend, bsum);
    pdl_trigger();
    {
        // the quad of a thread: outputs n0 + i .. i + 3 at reduction index r of the k-tile (QuadMap<false, UN, 1>): the 16
        // reduction indices of an output group meet through shared memory (the stage ring is free again)
        float (*sb)[UN] = reinterpret_cast<float (*)[UN]>(c.stages);
        if (want_bias && threadIdx.x < UT) {
            const QuadMap<false, UN, 1> mb;
#pragma unroll
            for (int e = 0; e < 4; ++e) sb[mb.r[0]][mb.i[0] + e] = bsum[0][e];
        }
        __syncthreads();
        if (want_bias && threadIdx.x < UN) {
            const float bmul = a.db_mul != 0.f ? a.db_mul : 1.0f;
            float v = 0.f;
#pragma unroll
            for (int r = 0; r < UK; ++r) v += sb[r][threadIdx.x];
            const int n = n0 + threadIdx.x;
            if (n < a.N) {
                if (part_b) part_b[(long long)blockIdx.z * a.N + n] = bmul * v;
                else atomicAdd(a.db + (long long)zb * a.db_bs + n, bmul * v);
            }
        }
    }
    float* dw = a.dw + (long long)zb * a.dw_bs;
    if (part && mbeg >= mend) {
        for (int idx = threadIdx.x; idx < UM * UN; idx += UTH) {
            const int k = k0 + idx % UM, n = n0 + idx / UM;
            if (n < a.N && k < K) part[((long long)blockIdx.z * a.N + n) * ldp + k] = 0.f;
        }
    }
    if (mbeg < mend)
        umma_epilogue(c, nsteps, [&](int i, int j, float (&v)[4]) {      // tile row i = k (a warp's lanes: 32 consecutive k), columns j .. j + 3 = n
            const int k = k0 + i;
            if (k >= K) return;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int n = n0 + j + e;
                if (n >= a.N) continue;
                if (part) part[((long long)blockIdx.z * a.N + n) * ldp + k] = v[e];
                else atomicAdd(dw + (long long)n * a.ldw + k, v[e]);
            }
        });
    umma_teardown(c, nsteps);
}

// second stage of the split weight gradient: fixed summation order.  blockDim = (32, 32): threadIdx.x walks 32 consecutive
// outputs (one coalesced 128-byte read per split), threadIdx.y deals the splits round-robin over 32 groups -- every thread has
// at most ceil(splits / 32) independent loads in flight, i.e. one memory round trip -- and one thread per output then adds the
// 32 group sums in group order: bitwise reproducible.
__global__ void __launch_bounds__(1024) wgrad_reduce_kernel(LinearWgrad a, int splits, int K, const float* part, const float* part_b, int ldp) {
    pdl_enter();
    __shared__ float acc[32][33];
    const int zb = blockIdx.y, g = threadIdx.y;
    const long long total = (long long)a.N * K + (part_b ? a.N : 0);
    for (long long base = (long long)blockIdx.x * 32; base < total; base += (long long)gridDim.x * 32) {
        const long long idx = base + threadIdx.x;
        float s = 0.f;
        bool is_b = false; int n = 0, k = 0;
        if (idx < total) {
            is_b = idx >= (long long)a.N * K;
            n = is_b ? (int)(idx - (long long)a.N * K) : (int)(idx / K);
            k = is_b ? 0 : (int)(idx % K);
            const float* src = is_b ? part_b + ((long long)zb * splits) * a.N + n : part + (((long long)zb * splits) * a.N + n) * ldp + k;
            const long long stride = is_b ? a.N : (long long)a.N * ldp;
            float s0 = 0.f, s1 = 0.f;
            int sp = g;
            for (; sp + 32 < splits; sp += 64) { s0 += src[sp * stride]; s1 += src[(sp + 32) * stride]; }
            if (sp < splits) s0 += src[sp * stride];
            s = s0 + s1;
        }
        acc[g][threadIdx.x] = s;
        __syncthreads();
        if (g == 0 && idx < total) {
            float t = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) t += acc[j][threadIdx.x];
            if (is_b) a.db[(long long)zb * a.db_bs + n] += t;
            else a.dw[(long long)zb * a.dw_bs + (long long)n * a.ldw + k] += t;
        }
        __syncthreads();
    }
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static int g_deterministic = -1;
// MARL_B200_WGRAD_SWAP=0: keep the default tile orientation everywhere (A/B switch)
static bool wgrad_swap_enabled() {
    static int on = -1;
    if (on < 0) { const char* e = getenv("MARL_B200_WGRAD_SWAP"); on = (e && e[0] == '0') ? 0 : 1; }
    return on == 1;
}
bool deterministic_wgrad() {
    if (g_deterministic < 0) { const char* e = getenv("MARL_B200_DETERMINISTIC"); g_deterministic = (e && e[0] == '1') ? 1 : 0; }
    return g_deterministic == 1;
}
void set_deterministic_wgrad(int on) { g_deterministic = on ? 1 : 0; }

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// 128-bit loads are legal when the base is 16-byte aligned and row pitch / region start are multiples of 4 floats
static bool vec_ok_lin(const LinOperand& o) {
    if (o.K1 == 0) return vec2_ok(o);      // only a second source (e.g. the shifted hidden state)
    return o.K1 >= 4 && o.x && aligned16(o.x) && (o.ldx & 3) == 0 && (o.K1 & 3) == 0 && ((o.x_bs & 3) == 0);
}
static bool vec_ok_mat(const float* p, int ld, long long bs, int col0 = 0) {
    return p && aligned16(p + col0) && (ld & 3) == 0 && ((bs & 3) == 0);
}

#define MARL_DISPATCH2(KERNEL, VA, VB, GRID, ST, ...)                                                      \
    do {                                                                                                   \
        static bool attr_done = false;                                                                     \
        if (!attr_done) {                                                                                  \
            cudaFuncSetAttribute(KERNEL<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem);   \
            cudaFuncSetAttribute(KERNEL<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem);  \
            cudaFuncSetAttribute(KERNEL<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem);  \
            cudaFuncSetAttribute(KERNEL<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem); \
            attr_done = true;                                                                              \
        }                                                                                                  \
        if (VA && VB) launch_pdl_prio(linear_prio(), KERNEL<true, true>, GRID, dim3(UTH), kUmmaSmem, ST, __VA_ARGS__);               \
        else if (VA) launch_pdl_prio(linear_prio(), KERNEL<true, false>, GRID, dim3(UTH), kUmmaSmem, ST, __VA_ARGS__);               \
        else if (VB) launch_pdl_prio(linear_prio(), KERNEL<false, true>, GRID, dim3(UTH), kUmmaSmem, ST, __VA_ARGS__);               \
        else launch_pdl_prio(linear_prio(), KERNEL<false, false>, GRID, dim3(UTH), kUmmaSmem, ST, __VA_ARGS__);                      \
    } while (0)

int linear_fwd(const LinearFwd& a, cudaStream_t st, bool tma) {
    if (a.M <= 0 || a.N <= 0 || a.batch <= 0) return MARL_OK;
    if (tma) { TGBuilder tg; if (tg.add_fwd(a)) return tg.launch(st); }       // TMA-addressable operands: tgemm.cu
    dim3 grid(cdiv(a.M, UM), cdiv(a.N, UN), a.batch);
    const bool va = vec_ok_lin(a.in), vb = vec_ok_mat(a.w, a.ldw, a.w_bs);
    { if (prof_enabled()) prof_note(a.M, a.N, lin_width(a.in)); ProfScope ps_("linear_fwd_kernel", st); MARL_DISPATCH2(linear_fwd_kernel, va, vb, grid, st, a); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

// 32 x 32 tiles through shared memory: coalesced on both sides
__global__ void __launch_bounds__(256) transpose_weights_kernel(const float* __restrict__ w, int ldw, int col0, int N, int K, float* __restrict__ wt, int ldwt) {
    pdl_enter();
    __shared__ float tile[32][33];
    const int n0 = blockIdx.x * 32, k0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int n = n0 + r, k = k0 + tx;
        tile[r][tx] = (n < N && k < K) ? __ldg(w + (long long)n * ldw + col0 + k) : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int k = k0 + r, n = n0 + tx;
        if (k < K && n < ldwt) wt[(long long)k * ldwt + n] = n < N ? tile[tx][r] : 0.f;
    }
}

int transpose_weights(const float* w, int ldw, int col0, int N, int K, float* wt, cudaStream_t st) {
    if (!w || !wt || N <= 0 || K <= 0) return MARL_EINVAL;
    ProfScope ps_("transpose_weights_kernel", st);
    launch_pdl_prio(linear_prio(), transpose_weights_kernel, dim3(cdiv(N, 32), cdiv(K, 32)), dim3(256), 0, st, w, ldw, col0, N, K, wt, transposed_pitch(N));
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

int linear_dgrad(const LinearDgrad& a, cudaStream_t st, bool tma) {
    if (a.M <= 0 || a.K <= 0 || a.batch <= 0) return MARL_OK;
    if (a.wt && a.batch != 1) return MARL_EINVAL;
    if (!a.wt && tma) { TGBuilder tg; if (tg.add_dgrad(a)) return tg.launch(st); }
    dim3 grid(cdiv(a.M, UM), cdiv(a.K, UN), a.batch);
    const bool va = vec_ok_mat(a.dy, a.lddy, a.dy_bs), vb = vec_ok_mat(a.w, a.ldw, a.w_bs, a.w_col0);
    if (a.wt) {
        static bool attr_done = false;
        if (!attr_done) {
            cudaFuncSetAttribute(linear_dgrad_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem);
            cudaFuncSetAttribute(linear_dgrad_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUmmaSmem);
            attr_done = true;
        }
        if (prof_enabled()) prof_note(a.M, a.K, a.N);
        ProfScope ps_("linear_dgrad_kernel", st);
        if (va) launch_pdl_prio(linear_prio(), linear_dgrad_kernel<true, true, true>, grid, dim3(UTH), kUmmaSmem, st, a);
        else launch_pdl_prio(linear_prio(), linear_dgrad_kernel<false, true, true>, grid, dim3(UTH), kUmmaSmem, st, a);
        MARL_LAUNCH_CHECK();
        return MARL_OK;
    }
    { if (prof_enabled()) prof_note(a.M, a.K, a.N); ProfScope ps_("linear_dgrad_kernel", st); MARL_DISPATCH2(linear_dgrad_kernel, va, vb, grid, st, a); }
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

int linear_wgrad(const LinearWgrad& a, cudaStream_t st, bool tma) {
    if (a.M <= 0 || a.N <= 0 || a.batch <= 0) return MARL_OK;
    if (tma) {
        TGBuilder tg;
        if (tg.add_wgrad(a)) { const int rc = tg.launch(st); return rc ? rc : tg.launch_reduce(st); }
    }
    const int K = lin_width(a.in);
    // tile orientation: outputs n along the 128 tile rows (default) or the input width k (linear_wgrad_swap_kernel), whichever
    // covers dw with fewer tiles
    // covers dw with fewer tiles -- provided the swapped grid still fills the machine: measured stand-alone (profiles/
    // r2c_gemm_linear.txt vs r2b_gemm_linear.txt) 153600 x 64 x 152: 165.6 -> 90.2 us, 5760 x 64 x 1232: 41.0 -> 24.4 us, but
    // 19200 x 64 x 192 (150 CTAs instead of 225): 17.7 -> 24.2 us, and config 2's fc1 (75 CTAs instead of 150) cost the step 10 us
    const int tiles_n = cdiv(a.N, UM) * cdiv(K, UN) * a.batch, tiles_s = cdiv(K, UM) * cdiv(a.N, UN) * a.batch;
    // rows per split of the swapped orientation (MARL_B200_WGRAD_SWAP_ROWS): 64 -- with one or two tiles the grid only fills the
    // machine when the reduction is cut finer than the 256 rows of the default orientation; config 2's fc1 gradient (1 tile x
    // 296 splits of 4 k-tiles instead of 2 tiles x 75 splits of 16) takes the step from 320 to 315 us (profiles/r2c_ab_swap_rows.txt;
    // 96 / 128 rows: 313 / 319 us; 48 / 32 rows with 3 / 4 CTAs per SM: 320 us; 128-row splits of the default orientation: no change)
    static int swap_rows = -1;
    if (swap_rows < 0) { const char* e = getenv("MARL_B200_WGRAD_SWAP_ROWS"); swap_rows = e ? atoi(e) : 64; if (swap_rows < 16) swap_rows = 64; }
    const int ctas_s = tiles_s * max(1, min(cdiv(2 * kNumSMs, tiles_s), cdiv(a.M, swap_rows)));
    const bool swap = kMnMajor && wgrad_swap_enabled() && tiles_s < tiles_n && 2 * ctas_s >= 3 * kNumSMs;
    const int tiles = swap ? tiles_s : tiles_n;
    int splits = cdiv(2 * kNumSMs, tiles);
    splits = max(1, min(splits, cdiv(a.M, swap ? swap_rows : 256)));   // 128 / 512 rows per split measured slower (r1d)
    int chunk = cdiv(cdiv(a.M, splits), UK) * UK;
    splits = cdiv(a.M, chunk);
    dim3 grid(swap ? cdiv(K, UM) : cdiv(a.N, UM), swap ? cdiv(a.N, UN) : cdiv(K, UN), a.batch * splits);
    const bool va = vec_ok_mat(a.dy, a.lddy, a.dy_bs), vb = vec_ok_lin(a.in);
    // deterministic path (marl_set_deterministic / MARL_B200_DETERMINISTIC=1; measured +13 us per weight gradient at the cfg-2
    // sizes, hence opt-in): per-split tiles in the scratch arena (marl_set_scratch) + a fixed-order reduce
    const int ldp = (K + 3) & ~3;
    const size_t pw = (size_t)a.batch * splits * a.N * ldp * sizeof(float), pb = a.db ? (size_t)a.batch * splits * a.N * sizeof(float) : 0;
    float* part = (splits * a.batch > 0 && deterministic_wgrad()) ? tgemm_scratch(pw + 256 + pb) : nullptr;
    float* part_b = (part && a.db) ? reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(part) + ((pw + 255) & ~(size_t)255)) : nullptr;
    if (swap) { if (prof_enabled()) prof_note(a.N, K, a.M); ProfScope ps_("linear_wgrad_kernel", st); MARL_DISPATCH2(linear_wgrad_swap_kernel, va, vb, grid, st, a, splits, chunk, part, part_b, ldp); }
    else { if (prof_enabled()) prof_note(a.N, K, a.M); ProfScope ps_("linear_wgrad_kernel", st); MARL_DISPATCH2(linear_wgrad_kernel, va, vb, grid, st, a, splits, chunk, part, part_b, ldp); }
    MARL_LAUNCH_CHECK();
    if (part) {
        const long long total = (long long)a.N * K + a.N;
        int bx = (int)((total + 31) / 32);
        if (bx > 4 * kNumSMs) bx = 4 * kNumSMs;
        // batched problems that accumulate into ONE dw (dw_bs == 0: e.g. the per-episode h0 term of dW_hh) are extra splits
        const bool fold = a.batch > 1 && a.dw_bs == 0 && (!a.db || a.db_bs == 0);
        ProfScope ps_("wgrad_reduce_kernel", st);
        launch_pdl_prio(linear_prio(), wgrad_reduce_kernel, dim3(bx, fold ? 1 : a.batch), dim3(32, 32), 0, st, a, fold ? splits * a.batch : splits, K,
                        (const float*)part, (const float*)part_b, ldp);
        MARL_LAUNCH_CHECK();
    }
    return MARL_OK;
}

}  // namespace marl
