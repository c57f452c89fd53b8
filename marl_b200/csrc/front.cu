// Input layers of the recurrent agent for ALL unrolls of a step in one persistent launch:
//     x  = relu(fc1([obs | last_action | agent_id]))      (network/q_network.py:17)
//     gi = W_ih x + b_ih                                  (the input half of the GRUCell, network/q_network.py:19)
// for every (episode, step, agent) row of every stream (eval on o, target on o_next, double-Q eval on o_next:
// controller/share_params.py:125-168).
//
// One CTA per SM walks 128-row tiles.  Roles (18 warps):
//   1 TMA warp         obs tile -> shared memory, 32 columns x 128 rows per box (cp.async.bulk.tensor, 128-byte swizzle), a ring
//                      of kRawSlots boxes in flight.  (The register-staged version of this kernel was bound by the LSU: ~1 us to
//                      ISSUE the loads of a k-tile behind the epilogue's stores, tools/front_trace.py.)
//   8 converter warps  thread = tile row (two groups alternate k-tiles): raw box (+ the last-action / agent-id columns, composed on the fly) -> hi / lo TF32
//                      halves -> TENSOR MEMORY (tcgen05.st), the A operand of GEMM 1; the k-tile's slice of W1 -> hi / lo in
//                      shared memory (B operand)
//   1 MMA warp         GEMM 1: acc1[128 x 64]  = in . W1^T     tcgen05.mma kind::tf32, A from TMEM
//                      GEMM 2: acc2[128 x 192] = x . W_ih^T    A from TMEM, B = W_ih resident in shared memory for the CTA's life
//   4 "E" warps        acc1 -> +b1 -> ReLU -> x split into hi / lo and written back to TMEM as GEMM 2's A; fp32 x -> global
//   4 "F" warps        acc2 -> +b_ih -> gi -> global
// Both outputs leave as 32 x 32 boxes through cp.async.bulk.tensor stores from 128-byte-swizzled staging blocks.  x never makes
// the round trip through HBM/L2 between the two layers, and the stages overlap across tiles.
//
// 3xTF32 (see linear.cu).  GEMM 1 streams its reduction, so the two 2^-11 correction products go to their own
// accumulator; GEMM 2 has both operands resident and issues ALL its correction products first: the accumulator is still
// ~2^-11 of its final magnitude while they land, so the fp32-accumulate truncation they add is negligible and the eight
// main products see the same number of updates as with a separate correction accumulator.
#include <cuda.h>
#include "front.h"
#include "umma.cuh"
#include "tgemm.h"
#include "profile.h"
#include "../../include/marl_b200.h"

namespace marl {

constexpr int FM = 128, FN1 = MARL_H, FN2 = MARL_G, FK = 16;
// E / converter / F warps: warp % 4 = TMEM lane quarter.  Two converter groups of four warps: group 0 takes the even k-tiles (A / B
// buffer 0), group 1 the odd ones (buffer 1)
constexpr int kWarpE = 0, kWarpC = 4, kWarpF = 12, kWarpMma = 16, kWarpTma = 17;
constexpr int kFrontThreads = 18 * 32;
constexpr int FB_PITCH = FN1 * 4 + 8, FW_PITCH = FN2 * 4 + 8;   // canonical K-major layout, see linear.cu
#ifndef MARL_FRONT_SLOTS
#define MARL_FRONT_SLOTS 3
#endif
constexpr int kRawSlots = MARL_FRONT_SLOTS;                     // obs boxes in flight per CTA (16 KB each)
constexpr int kBoxCols = 2 * FK;                                // one box = two k-tiles: 128-byte rows = whole L2 lines
constexpr int kRawBytes = FM * kBoxCols * 4;

// TMEM columns
constexpr uint32_t kColAcc1 = 0, kColCorr1 = 64, kColXhi = 128, kColXlo = 192, kColAcc2 = 256, kColA = 448, kFrontTmemCols = 512;

struct FrontB {                                                  // one k-tile of W1, hi / lo
    float hi[(FK / 4) * FB_PITCH];
    float lo[(FK / 4) * FB_PITCH];
};

struct alignas(1024) FrontSmem {
    unsigned char raw[kRawSlots][kRawBytes];                     // TMA boxes [128 rows][128 B], 128-byte swizzle
    float stage_e[4][32 * 32];                                   // per E warp: one swizzled 32 x 32 box of x (columns 0-31, then 32-63)
    float stage_f[4][2][32 * 32];                                // per F warp: two gi boxes (one draining, one being filled)
    float wih_hi[(MARL_H / 4) * FW_PITCH];
    float wih_lo[(MARL_H / 4) * FW_PITCH];
    FrontB b[2];
    float b1[FN1];
    float bih[FN2];
    FrontSet set;
    FrontStream s[kFrontMaxStreams];
    uint64_t raw_full[kRawSlots], raw_empty[kRawSlots];
    uint64_t a_full[2], a_empty[2];
    uint64_t acc1_full, acc1_free, xa_ready, acc2_full, acc2_free;
    uint32_t tmem_base;
};
constexpr size_t kFrontSmemBytes = sizeof(FrontSmem) + 1024;
static_assert(kFrontSmemBytes <= 227 * 1024, "front kernel shared memory");

constexpr uint32_t front_idesc(int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(FM >> 4) << 24); }

__device__ __forceinline__ void fmma_ts(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(d), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void fcommit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int c0, int c1, const void* src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(map), "r"(c0), "r"(c1), "r"(smem_u32(src)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                   "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// debug phase trace of CTA 0: (tag, globaltimer ns) pairs, 255 per role (0 converter, 1 MMA, 2 E, 3 F)
#define FT_STAMP(role, tag)                                                                                            \
    do {                                                                                                               \
        if (trace && tn < 255) {                                                                                       \
            long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                       \
            trace[(role) * 512 + 2 * tn] = (tag); trace[(role) * 512 + 2 * tn + 1] = t_; ++tn; trace[(role) * 512 + 510] = tn; \
        }                                                                                                              \
    } while (0)

struct FrontMaps {
    CUtensorMap obs[kFrontMaxStreams];      // [rows, K1]   box {32, 128}, 128-byte swizzle
    CUtensorMap x[kFrontMaxStreams];        // [rows, 64]   box {32, 32}, 128-byte swizzle
    CUtensorMap gi[kFrontMaxStreams];       // [rows, 192]  box {32, 32}, 128-byte swizzle
};

__global__ void __launch_bounds__(kFrontThreads, 1) agent_front_kernel(const FrontArgs a, const __grid_constant__ FrontMaps maps) {
    extern __shared__ unsigned char front_smem_raw[];
    FrontSmem& sm = *reinterpret_cast<FrontSmem*>((reinterpret_cast<uintptr_t>(front_smem_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int role = warp == kWarpC ? 0 : warp == kWarpMma ? 1 : warp == kWarpE ? 2 : warp == kWarpF ? 3 : 0;
    long long* trace = (blockIdx.x == 0 && lane == 0 && (warp == kWarpC || warp == kWarpMma || warp == kWarpE || warp == kWarpF)) ? a.trace : nullptr;
    int tn = 0;

    // ---- which parameter set this CTA serves, copied to shared memory (dynamically indexed reads of the kernel
    // parameter bank cost ~200 cycles each)
    int p = 0;
    for (int k = 1; k < a.n_sets; ++k) if ((int)blockIdx.x >= a.set[k].cta0) p = k;
    if (tid == 0) {
        sm.set = a.set[p];
        for (int k = 0; k < kFrontMaxStreams; ++k) sm.s[k] = a.s[k];
#pragma unroll
        for (int s = 0; s < kRawSlots; ++s) { mbar_init(&sm.raw_full[s], 1); mbar_init(&sm.raw_empty[s], 256); }
#pragma unroll
        for (int s = 0; s < 2; ++s) { mbar_init(&sm.a_full[s], 128); mbar_init(&sm.a_empty[s], 1); }
        mbar_init(&sm.acc1_full, 1); mbar_init(&sm.acc1_free, 128); mbar_init(&sm.xa_ready, 128);
        mbar_init(&sm.acc2_full, 1); mbar_init(&sm.acc2_free, 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarpMma) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(kFrontTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    FT_STAMP(role, 9000);
    pdl_wait();                                          // nothing above touched global memory
    FT_STAMP(role, 9001);
    const uint32_t tmem = sm.tmem_base;
    const int I = a.I, rows = a.rows, tps = a.tiles_per_stream;
    const int nk = (I + FK - 1) / FK;
    const int n_ctas = sm.set.n_ctas, cta = (int)blockIdx.x - sm.set.cta0;
    const int set_tiles = sm.set.n_streams * tps;
    const int n_my = cta < set_tiles ? (set_tiles - cta + n_ctas - 1) / n_ctas : 0;
    const int nb = (nk + 1) / 2;                         // boxes per tile: box j holds k-tiles 2j (converter group 0) and 2j + 1 (group 1)
    const int total_boxes = n_my * nb;

    // =========================================================== TMA producer (lane 0 of its warp)
    int tma_it = 0, tma_j = 0;
    auto tma_issue = [&](int b_begin, int b_end) {
        for (int bs = b_begin; bs < b_end; ++bs) {
            const int r = bs % kRawSlots, use = bs / kRawSlots;
            mbar_wait(&sm.raw_empty[r], (uint32_t)((use & 1) ^ 1));
            const int t = cta + tma_it * n_ctas, si = sm.set.stream[t / tps];
            if (tma_j * kBoxCols < sm.s[si].in.K1) {
                mbar_expect_tx(&sm.raw_full[r], (uint32_t)kRawBytes);      // (columns / rows past the tensor are zero-filled and counted)
                tma_load_2d(sm.raw[r], &maps.obs[si], tma_j * kBoxCols, (t % tps) * FM, &sm.raw_full[r]);
            } else {
                mbar_arrive(&sm.raw_full[r]);                              // a box made of composed columns only
            }
            if (++tma_j == nb) { tma_j = 0; ++tma_it; }
        }
    };
    const int tma_prologue = total_boxes < kRawSlots ? total_boxes : kRawSlots;
    if (warp == kWarpTma) {
        if (lane == 0) tma_issue(0, tma_prologue);      // the first boxes are in flight while the other warps stage the weights
        __syncwarp();
    } else {
        // ---- resident operands: W_ih as hi / lo TF32 halves in the K-major UMMA layout, the two bias vectors
        const float* w = sm.set.w_ih;
        for (int idx = tid; idx < FN2 * (MARL_H / 4); idx += kWarpTma * 32) {
            const int n = idx >> 4, c = idx & 15;
            const float4 v = __ldg(reinterpret_cast<const float4*>(w + (long long)n * MARL_H + 4 * c));
            float4 h, l;
            tf32_split(v.x, h.x, l.x); tf32_split(v.y, h.y, l.y); tf32_split(v.z, h.z, l.z); tf32_split(v.w, h.w, l.w);
            *reinterpret_cast<float4*>(sm.wih_hi + c * FW_PITCH + n * 4) = h;
            *reinterpret_cast<float4*>(sm.wih_lo + c * FW_PITCH + n * 4) = l;
        }
        if (sm.set.w_ih_t) {
            // W_ih^T for the data gradient of this step's backward pass: each CTA of the set writes its slice
            const int total_e = FN2 * MARL_H, per = (total_e + n_ctas - 1) / n_ctas;
            const int e0 = cta * per, e1 = min(total_e, e0 + per);
            for (int e = e0 + tid; e < e1; e += kWarpTma * 32) {
                const int k = e / FN2, n = e - k * FN2;                   // consecutive threads: consecutive n of one row of W_ih^T
                sm.set.w_ih_t[e] = __ldg(w + (long long)n * MARL_H + k);
            }
        }
        if (tid < FN1) sm.b1[tid] = sm.set.b1 ? __ldg(sm.set.b1 + tid) : 0.f;
        if (tid < FN2) sm.bih[tid] = sm.set.b_ih ? __ldg(sm.set.b_ih + tid) : 0.f;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    FT_STAMP(role, 9002);

    if (warp >= kWarpC && warp < kWarpF) {
        // =========================================================== converters: thread = tile row, group = k-tile parity
        const int grp = (warp - kWarpC) >> 2;                                              // k-tiles g = grp, grp + 2, ...
        const int q = warp & 3, row_in_tile = q * 32 + lane, ct = (tid - kWarpC * 32) & 127;   // ct: 0..127 inside the group
        const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);
        // this thread's two quads of the W1 k-tile: feature row bj, 16-byte chunk bc
        const int bj[2] = {ct >> 2, (ct + 128) >> 2}, bc = ct & 3;
        const OpMat B{sm.set.w1, I, FN1, I, sm.set.vec_w1 != 0};
        const OpMat::Row brow[2] = {B.row(bj[0]), B.row(bj[1])};
        float4 wq[2];
        auto load_w1 = [&](int kt) {                                                       // W1 slice of a k-tile (L2-resident)
            const int kn = kt * FK + 4 * bc;
            wq[0] = kn < I ? B.quad_at(brow[0], kn) : make_float4(0.f, 0.f, 0.f, 0.f);
            wq[1] = kn < I ? B.quad_at(brow[1], kn) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        load_w1(grp < nk ? grp : 0);
        // row context of the composed columns [K1, I): last action (shifted one step inside the episode) and agent id
        const float* x2r = nullptr; int hot = -1, K1 = 0, K2 = 0;
        const int bsel = grp;
        int use = 0, it = 0, j = 0;
        for (int bs = 0; bs < total_boxes; ++bs) {
            const int r = bs % kRawSlots, kt = 2 * j + grp;
            const uint32_t box_parity = (uint32_t)((bs / kRawSlots) & 1);
            if (j == 0) {
                const int t = cta + it * n_ctas;
                const LinOperand& o = sm.s[sm.set.stream[t / tps]].in;
                const int m = (t % tps) * FM + row_in_tile;
                K1 = o.K1; K2 = o.K2; x2r = nullptr; hot = -1;
                if (m < rows) {
                    if (K2 > 0 && !(o.x2_shift && (m % o.x2_period) < o.x2_shift)) x2r = o.x2 + (long long)(m - o.x2_shift) * o.ldx2;
                    if (o.onehot_mod) hot = K1 + K2 + (m % o.onehot_mod);
                }
            }
            const int jn = (j + 1 == nb) ? 0 : j + 1;
            if (kt >= nk) {                                                   // odd number of k-tiles: the last box has no second half
                mbar_wait(&sm.raw_full[r], box_parity);
                mbar_arrive(&sm.raw_empty[r]);
                j = jn; if (j == 0) ++it;
                continue;
            }
            const int k0 = kt * FK;
            float v[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = 0.f;
            // the composed columns first (global loads in flight while the box is awaited)
            if (k0 + FK > K1) {
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int k = k0 + e;
                    if (k >= K1 && k < K1 + K2) { if (x2r) v[e] = __ldg(x2r + (k - K1)); }
                    else if (k == hot) v[e] = 1.0f;
                }
            }
            mbar_wait(&sm.raw_full[r], box_parity);
            if (k0 < K1) {
                // 128-byte swizzle: 16-byte chunk c of box row rr sits at chunk c ^ (rr & 7); this group's k-tile = chunks 4 grp ..
                const unsigned char* box = sm.raw[r] + row_in_tile * 128;
                const int sw = row_in_tile & 7;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 t4 = *reinterpret_cast<const float4*>(box + (((4 * grp + c) ^ sw) << 4));
                    if (k0 + 4 * c + 3 < K1) { v[4 * c] = t4.x; v[4 * c + 1] = t4.y; v[4 * c + 2] = t4.z; v[4 * c + 3] = t4.w; }
                    else {
                        if (k0 + 4 * c < K1) v[4 * c] = t4.x;
                        if (k0 + 4 * c + 1 < K1) v[4 * c + 1] = t4.y;
                        if (k0 + 4 * c + 2 < K1) v[4 * c + 2] = t4.z;
                    }
                }
            }
            mbar_arrive(&sm.raw_empty[r]);                                   // (values are in registers)
            uint32_t h[16], l[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                float hh, ll;
                tf32_split(v[e], hh, ll);
                h[e] = __float_as_uint(hh); l[e] = __float_as_uint(ll);
            }
            mbar_wait(&sm.a_empty[bsel], (uint32_t)((use & 1) ^ 1));         // the MMAs that read this A / B buffer pair are done
            tc_fence_after();
            FT_STAMP(0, bs);
            tmem_st16(tq + kColA + 32 * bsel, h);
            tmem_st16(tq + kColA + 32 * bsel + 16, l);
            FrontB& sb = sm.b[bsel];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                float4 hh, ll;
                tf32_split(wq[u].x, hh.x, ll.x); tf32_split(wq[u].y, hh.y, ll.y); tf32_split(wq[u].z, hh.z, ll.z); tf32_split(wq[u].w, hh.w, ll.w);
                *reinterpret_cast<float4*>(sb.hi + bc * FB_PITCH + bj[u] * 4) = hh;
                *reinterpret_cast<float4*>(sb.lo + bc * FB_PITCH + bj[u] * 4) = ll;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(&sm.a_full[bsel]);
            FT_STAMP(0, 1000 + bs);
            ++use;
            j = jn; if (j == 0) ++it;
            load_w1(2 * j + grp < nk ? 2 * j + grp : grp);                    // this group's next k-tile
        }
    } else if (warp == kWarpMma) {
        // =========================================================== MMA issue (lane 0)
        const uint32_t id1 = front_idesc(FN1), id2 = front_idesc(FN2);
        for (int it = 0; it < n_my; ++it) {
            mbar_wait(&sm.acc1_free, (uint32_t)((it & 1) ^ 1));            // x(it-1) has been read out of acc1
            tc_fence_after();
            for (int kt = 0; kt < nk; ++kt) {
                const int bsel = kt & 1;                                   // converter group = k-tile parity inside the tile
                const int use = (bsel ? it * (nk >> 1) : it * nb) + (kt >> 1);
                mbar_wait(&sm.a_full[bsel], (uint32_t)(use & 1));
                tc_fence_after();
                FT_STAMP(1, it * nk + kt);
                if (lane == 0) {
                    const FrontB& sb = sm.b[bsel];
                    const uint32_t ta = tmem + kColA + 32 * bsel;
#pragma unroll
                    for (int k8 = 0; k8 < FK / 8; ++k8) {
                        const uint32_t bo = (uint32_t)(2 * k8) * FB_PITCH * 4;
                        const uint64_t dbh = umma_desc(smem_u32(sb.hi) + bo, FB_PITCH * 4, 128), dbl = umma_desc(smem_u32(sb.lo) + bo, FB_PITCH * 4, 128);
                        const uint32_t first = (kt | k8) ? 1u : 0u;
                        fmma_ts(tmem + kColCorr1, ta + 16 + 8 * k8, dbh, id1, first);      // lo . hi
                        fmma_ts(tmem + kColCorr1, ta + 8 * k8, dbl, id1, 1u);              // hi . lo
                        fmma_ts(tmem + kColAcc1, ta + 8 * k8, dbh, id1, first);            // hi . hi
                    }
                    fcommit(&sm.a_empty[bsel]);
                    if (kt == nk - 1) fcommit(&sm.acc1_full);
                }
                __syncwarp();
            }
            // GEMM 2 of this tile
            mbar_wait(&sm.xa_ready, (uint32_t)(it & 1));                   // x(it) hi / lo are in TMEM
            mbar_wait(&sm.acc2_free, (uint32_t)((it & 1) ^ 1));            // gi(it-1) has been read out of acc2
            tc_fence_after();
            FT_STAMP(1, 2000 + it);
            if (lane == 0) {
                const uint32_t wh = smem_u32(sm.wih_hi), wl = smem_u32(sm.wih_lo);
#pragma unroll
                for (int k8 = 0; k8 < MARL_H / 8; ++k8) {
                    const uint32_t bo = (uint32_t)(2 * k8) * FW_PITCH * 4;
                    fmma_ts(tmem + kColAcc2, tmem + kColXlo + 8 * k8, umma_desc(wh + bo, FW_PITCH * 4, 128), id2, k8 ? 1u : 0u);
                    fmma_ts(tmem + kColAcc2, tmem + kColXhi + 8 * k8, umma_desc(wl + bo, FW_PITCH * 4, 128), id2, 1u);
                }
#pragma unroll
                for (int k8 = 0; k8 < MARL_H / 8; ++k8) {
                    const uint32_t bo = (uint32_t)(2 * k8) * FW_PITCH * 4;
                    fmma_ts(tmem + kColAcc2, tmem + kColXhi + 8 * k8, umma_desc(wh + bo, FW_PITCH * 4, 128), id2, 1u);
                }
                fcommit(&sm.acc2_full);
            }
            FT_STAMP(1, 3000 + it);
            __syncwarp();
        }
    } else if (warp < kWarpC) {
        // =========================================================== E: acc1 -> x -> (TMEM hi/lo, global)
        const int q = warp & 3;                                            // TMEM lane quarter this warp may touch
        const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);
        float* blk = &sm.stage_e[q][0];
        for (int it = 0; it < n_my; ++it) {
            const int t = cta + it * n_ctas, si = sm.set.stream[t / tps];
            const bool store_x = sm.s[si].store_x != 0;
            const int m0 = (t % tps) * FM;
            mbar_wait(&sm.acc1_full, (uint32_t)(it & 1));
            FT_STAMP(2, it);
            if (it > 0) mbar_wait(&sm.acc2_full, (uint32_t)((it - 1) & 1));   // GEMM 2 of the previous tile has read x(it-1) from TMEM
            tc_fence_after();
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the last box of the previous tile has left the staging block
            __syncwarp();
            // 16 columns at a time: acc1 -> +b1 -> ReLU -> hi / lo back into TMEM.  The fp32 values of columns 0-31 are parked in
            // the warp's staging box (lane = row, 16-byte chunk ch at ch ^ (row & 7): conflict-free), those of columns 32-63 in
            // registers; both leave AFTER the hand-over, off the MMA warp's critical path
            float keep[32];
#pragma unroll
            for (int c = 0; c < FN1 / 16; ++c) {
                uint32_t m[16], k[16];
                tmem_ld16(tq + kColAcc1 + 16 * c, m);
                tmem_ld16(tq + kColCorr1 + 16 * c, k);
                tmem_wait_ld();
#pragma unroll
                for (int e4 = 0; e4 < 16; e4 += 4) {
                    float xv[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        xv[e] = fmaxf(__uint_as_float(m[e4 + e]) + __uint_as_float(k[e4 + e]) + sm.b1[16 * c + e4 + e], 0.f);
                        float hh, ll;
                        tf32_split(xv[e], hh, ll);
                        m[e4 + e] = __float_as_uint(hh); k[e4 + e] = __float_as_uint(ll);
                    }
                    if (c < 2) {
                        const int ch = c * 4 + (e4 >> 2);
                        if (store_x) *reinterpret_cast<float4*>(blk + lane * 32 + 4 * (ch ^ (lane & 7))) = make_float4(xv[0], xv[1], xv[2], xv[3]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) keep[(c - 2) * 16 + e4 + e] = xv[e];
                    }
                }
                tmem_st16(tq + kColXhi + 16 * c, m);
                tmem_st16(tq + kColXlo + 16 * c, k);
            }
            tc_fence_before();
            mbar_arrive(&sm.acc1_free);
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(&sm.xa_ready);
            FT_STAMP(2, 1000 + it);
            if (store_x) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&maps.x[si], 0, m0 + q * 32, blk);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                }
                __syncwarp();
#pragma unroll
                for (int ch = 0; ch < 8; ++ch)
                    *reinterpret_cast<float4*>(blk + lane * 32 + 4 * (ch ^ (lane & 7))) = make_float4(keep[4 * ch], keep[4 * ch + 1], keep[4 * ch + 2], keep[4 * ch + 3]);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&maps.x[si], 32, m0 + q * 32, blk);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            FT_STAMP(2, 2000 + it);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else if (warp == kWarpTma) {
        if (lane == 0) tma_issue(tma_prologue, total_boxes);
        __syncwarp();
    } else if (warp < kWarpMma) {
        // =========================================================== F: acc2 -> gi
        const int q = warp & 3;
        const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);
        int seq = 0;
        for (int it = 0; it < n_my; ++it) {
            const int t = cta + it * n_ctas, si = sm.set.stream[t / tps];
            const int m0 = (t % tps) * FM;
            mbar_wait(&sm.acc2_full, (uint32_t)(it & 1));
            tc_fence_after();
            FT_STAMP(3, it);
#pragma unroll 1
            for (int c = 0; c < FN2 / 32; ++c, ++seq) {
                uint32_t v[32];
                tmem_ld32(tq + kColAcc2 + 32 * c, v);
                float* blk = &sm.stage_f[q][seq & 1][0];
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store that last used this block has read it
                __syncwarp();
                tmem_wait_ld();
                if (c == FN2 / 32 - 1) { tc_fence_before(); mbar_arrive(&sm.acc2_free); }
#pragma unroll
                for (int g4 = 0; g4 < 8; ++g4) {
                    const float4 b = *reinterpret_cast<const float4*>(&sm.bih[32 * c + 4 * g4]);
                    *reinterpret_cast<float4*>(blk + lane * 32 + 4 * (g4 ^ (lane & 7))) =
                        make_float4(__uint_as_float(v[4 * g4]) + b.x, __uint_as_float(v[4 * g4 + 1]) + b.y,
                                    __uint_as_float(v[4 * g4 + 2]) + b.z, __uint_as_float(v[4 * g4 + 3]) + b.w);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&maps.gi[si], 32 * c, m0 + q * 32, blk);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            FT_STAMP(3, 1000 + it);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    FT_STAMP(role, 9003);
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    if (warp == kWarpMma) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kFrontTmemCols));
}

static int g_front_on = -1;
bool front_enabled() {
    if (g_front_on < 0) { const char* e = getenv("MARL_B200_FRONT"); g_front_on = (e && e[0] == '0') ? 0 : 1; }
    return g_front_on == 1;
}

namespace {

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

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
// 2-D fp32 tensor [rows, cols] with a row pitch in floats
bool make_map(CUtensorMap* m, const float* base, int cols, long long rows, long long pitch, int box_c, int box_r, CUtensorMapSwizzle sw) {
    EncodeTiled enc = encoder();
    if (!enc || !base || !aligned16(base) || (pitch & 3) || cols <= 0 || rows <= 0) return false;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)pitch * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_c, (cuuint32_t)box_r};
    cuuint32_t est[2] = {1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, est, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

// Groups the streams into parameter sets and deals the CTAs of the grid to the sets in proportion to their tiles.
// a.s[0 .. n_streams), a.rows, a.I are filled by the caller, together with one FrontSet per stream in a.set[i]
// (w1 / b1 / w_ih / b_ih of stream i); this merges equal sets.
// budget > 0: at most that many CTAs, and every set keeps only as many as its fullest CTA's tile count needs -- a launch that
// shares the machine with another one (marl_agent_unroll_fwd's split forward) leaves the SMs it could not use to the other.
bool front_plan(FrontArgs& a, int n_streams, int budget) {
    if (!front_enabled() || !encoder() || n_streams < 1 || n_streams > kFrontMaxStreams || a.rows <= 0) return false;
    if (a.I <= 0 || a.I > 256) return false;            // GEMM 1 keeps one main accumulator: <= 32 accumulator updates
    if (a.hidden != MARL_H) return false;               // x [rows, 64], gi [rows, 192] and the W_ih staging are 64-wide
    for (int i = 0; i < n_streams; ++i) {
        if (!aligned16(a.s[i].gi) || !a.s[i].x || !aligned16(a.s[i].x)) return false;
        if (!aligned16(a.set[i].w_ih)) return false;
        const LinOperand& o = a.s[i].in;
        // the first source goes through a tensor map: dense 16-byte-aligned rows
        if (o.K1 <= 0 || !o.x || !aligned16(o.x) || (o.ldx & 3) || o.x_bs != 0) return false;
        if (lin_width(o) != a.I) return false;
        a.s[i].vec_in = 1;
        a.set[i].vec_w1 = aligned16(a.set[i].w1) && (a.I & 3) == 0;
    }
    FrontSet sets[kFrontMaxStreams];
    int ns = 0;
    for (int i = 0; i < n_streams; ++i) {
        int hit = -1;
        for (int k = 0; k < ns; ++k)
            if (sets[k].w1 == a.set[i].w1 && sets[k].b1 == a.set[i].b1 && sets[k].w_ih == a.set[i].w_ih && sets[k].b_ih == a.set[i].b_ih) hit = k;
        if (hit < 0) { sets[ns] = a.set[i]; sets[ns].n_streams = 0; hit = ns++; }
        else if (a.set[i].w_ih_t) sets[hit].w_ih_t = a.set[i].w_ih_t;
        sets[hit].stream[sets[hit].n_streams++] = i;
    }
    a.tiles_per_stream = (a.rows + FM - 1) / FM;
    const long long total = (long long)n_streams * a.tiles_per_stream;
    const int cap = budget > 0 && budget < kNumSMs ? budget : kNumSMs;
    if (cap < ns) return false;
    const int grid = (int)(total < cap ? total : cap);
    int ctas[kFrontMaxStreams];
    for (int k = 0; k < ns; ++k) ctas[k] = 1;
    for (int left = grid - ns; left > 0; --left) {       // the next CTA goes to the set with the most tiles per CTA
        int best = 0;
        for (int k = 1; k < ns; ++k)
            if ((double)sets[k].n_streams / ctas[k] > (double)sets[best].n_streams / ctas[best]) best = k;
        ++ctas[best];
    }
    if (budget > 0)
        for (int k = 0; k < ns; ++k) {                   // fewest CTAs at the same tiles per CTA (150 tiles on 80 CTAs: 75 x 2)
            const int t = sets[k].n_streams * a.tiles_per_stream, per = (t + ctas[k] - 1) / ctas[k];
            ctas[k] = (t + per - 1) / per;
        }
    int c0 = 0;
    for (int k = 0; k < ns; ++k) { sets[k].cta0 = c0; sets[k].n_ctas = ctas[k]; c0 += ctas[k]; a.set[k] = sets[k]; }
    a.n_sets = ns;
    return true;
}

int front_launch(const FrontArgs& a, int n_streams, int prio, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) { cudaFuncSetAttribute(agent_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFrontSmemBytes); attr_set = true; }
    FrontMaps maps;
    for (int i = 0; i < kFrontMaxStreams; ++i) {
        const FrontStream& S = a.s[i < n_streams ? i : 0];
        if (!make_map(&maps.obs[i], S.in.x, S.in.K1, a.rows, S.in.ldx, kBoxCols, FM, CU_TENSOR_MAP_SWIZZLE_128B)) return MARL_EINVAL;
        if (!make_map(&maps.x[i], S.x, FN1, a.rows, FN1, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return MARL_EINVAL;
        if (!make_map(&maps.gi[i], S.gi, FN2, a.rows, FN2, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B)) return MARL_EINVAL;
    }
    int grid = 0;
    for (int k = 0; k < a.n_sets; ++k) grid += a.set[k].n_ctas;
    ProfScope ps_("agent_front_kernel", st);
    FrontArgs b = a;
    b.trace = trace_buffer();
    launch_pdl_prio(prio, agent_front_kernel, dim3(grid), dim3(kFrontThreads), kFrontSmemBytes, st, b, maps);
    MARL_LAUNCH_CHECK();
    return MARL_OK;
}

}  // namespace marl

// on = 0: the input layers run as separate launches (linear.cu) -- the A/B switch behind MARL_B200_FRONT; returns the previous setting
extern "C" int marl_front_enable(int on) {
    const int prev = marl::front_enabled() ? 1 : 0;
    marl::g_front_on = on ? 1 : 0;
    return prev;
}
