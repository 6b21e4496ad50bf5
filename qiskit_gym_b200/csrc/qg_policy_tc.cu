// qg_policy_tc.cu — the policy network for LARGE batches (the rollout collector at 65 536 environments) on the 5th-generation tensor
// cores: tcgen05.mma with accumulators in tensor memory, operands streamed into shared memory by bulk copies (cp.async.bulk, the TMA
// unit's 1-D form) that complete on mbarriers, tcgen05.ld epilogues.  SURVEY.md §8f row 3 at collector scale; the small-batch search
// keeps the f32 FFMA kernel of qg_policy_kernels.cuh (8 rows per CTA is latency-, not throughput-bound).
//
// Arithmetic.  A twisterl BasicPolicy is Linear -> ReLU chains in f32.  To stay within the 1e-4 logit tolerance of the f32 module on
// f16 tensor-core inputs, every f32 value v is carried as two halves  v ~ hi + lo,  hi = half(v), lo = half(v - hi)  (22 significant bits) and
// a product is evaluated as  a_hi*w_hi + a_hi*w_lo + a_lo*w_hi  with f32 accumulation in tensor memory (the dropped lo*lo term is 2^-22
// relative).  The first layer's input is 0/1 — exact in one half — so it needs two products, the others three.
//
// One kernel per layer:  Y[128-row tile][NT columns] = act(X W^T + b),  persistent CTAs looping over (row tile, column tile) pairs,
//   warp 0  loader  : one lane issues the stage's bulk copies (X tile images written by the previous layer's epilogue, W tile images laid
//                     out once at creation), 3 stages in flight, full / empty mbarriers;
//   warp 1  MMA     : one lane issues  tcgen05.mma.cta_group::1.kind::f16  M = 128, N = NT, K = 16  over the stage's 64-wide K block and
//                     commits the stage back to the loader (tcgen05.commit -> empty barrier) and, after the last K block, the accumulator to
//                     the epilogue; two accumulator buffers in tensor memory, so tile i+1's products overlap tile i's epilogue;
//   warps 2-5 epilogue: thread = output row (tensor-memory lane): tcgen05.ld 16 columns at a time, + bias, ReLU, split into halves, written as
//                     the next layer's X tile image (coalesced 16-byte stores); the last layer writes logits / softmax / value instead.
// Operand images use the no-swizzle K-major canonical layout  [k / 8][row][k % 8]  (8-row x 16-byte core matrices contiguous; leading
// byte offset = rows * 16 between the two 8-wide K chunks of one MMA, stride byte offset = 128 between 8-row groups), which is also the
// layout in which one epilogue thread per row writes 16 bytes per 8 columns with consecutive threads at consecutive addresses.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "qg_host.hpp"

namespace qg {
namespace tc {

constexpr int kM = 128;              // rows per tile (UMMA M, tensor-memory lanes)
constexpr int kKB = 64;              // K block (halves) per pipeline stage
constexpr int kStages = 3;
constexpr int kMaxNT = 128;          // widest column tile
constexpr int kThreads = 192;        // 6 warps: loader, MMA, 4 epilogue
constexpr int kImgA = kM * kKB;      // halves per X tile image (16 KB)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n .reg .pred p;\n"
        "TC_WAIT_LOOP:\n"
        " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        " @p bra TC_WAIT_DONE;\n"
        " bra TC_WAIT_LOOP;\n"
        "TC_WAIT_DONE:\n}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
#ifdef QG_TC_PROBE           // tools build: cycles the fused kernel's MMA-issuing thread and its epilogue warp 2 spend per class of work (qg_policy_tc_debug_read*)
__device__ long long g_tc_wait[160 * 8];     // waits on d1_empty, full (layer 1), a0_full, d2_empty, act_full (layer 2), full (layers 2 / 3), act_full (layer 3); total
__device__ long long g_tc_epi[160 * 8];      // waits d1_full, act_empty; convert (layer 1); wait d2_full; layer-2 pieces; head wait; head (with its wait); total
#define TC_MMA_WAIT(cls, bar, par) do { const long long _t0 = clock64(); mbar_wait(bar, par); tcw[cls] += clock64() - _t0; } while (0)
#define TC_EPI(cls, stmt) do { const long long _t0 = clock64(); stmt; tce[cls] += clock64() - _t0; } while (0)
#else
#define TC_MMA_WAIT(cls, bar, par) mbar_wait(bar, par)
#define TC_EPI(cls, stmt) do { stmt; } while (0)
#endif
__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes),
                 "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem]^T, f16 inputs, f32 accumulate (tcgen05.mma), and tcgen05.commit: all MMAs issued so far by the issuing
// thread arrive on the mbarrier when they have completed (implies tcgen05.fence::before_thread_sync) —
// for a whole converged warp: every lane runs the issue loop with warp-uniform operands and one elected lane (always the same
// one for the full mask) issues.  Under `if (lane == 0)` the compiler cannot tell that one lane is active and wraps every tcgen05.mma in a loop
// that broadcasts its operands into uniform registers (ELECT / 5 x R2UR.BROADCAST / BRA.U.ANY): ~20 instructions and ~115 cycles per MMA in
// the fused kernel, more than a 64-cycle layer-1 product takes on the tensor pipe (cuobjdump -sass, profiles/r2_v36_tc_probe.json).
__device__ __forceinline__ void umma_f16_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p, q;\n"
        " setp.ne.b32 p, %4, 0;\n"
        " elect.sync _|q, 0xffffffff;\n"
        " @q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// ... with the descriptors as their low words only (start address and leading byte offset; the high word — stride byte offset 128, version
// 1 — is the same for every operand of the fused kernel): stepping to the next K = 16 slice is one 32-bit add per operand
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return (saddr >> 4) | ((lbo_bytes >> 4) << 16); }
__device__ __forceinline__ void umma_f16_lo(uint32_t tmem_d, uint32_t alo, uint32_t blo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p, q;\n .reg .b32 hi;\n .reg .b64 ad, bd;\n"
        " setp.ne.b32 p, %4, 0;\n"
        " mov.u32 hi, 0x4008;\n"
        " mov.b64 ad, {%1, hi};\n"
        " mov.b64 bd, {%2, hi};\n"
        " elect.sync _|q, 0xffffffff;\n"
        " @q tcgen05.mma.cta_group::1.kind::f16 [%0], ad, bd, %3, p;\n}\n" ::"r"(tmem_d), "r"(alo), "r"(blo), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_w(uint64_t* bar) {
    asm volatile(
        "{\n .reg .pred q;\n"
        " elect.sync _|q, 0xffffffff;\n"
        " @q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                   "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor: start address, leading / stride byte offsets in 16-byte
// units, version 1 = sm_100, layout type 0)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): f32 accumulator, f16 A and B, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t instr_desc(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kM >> 4) << 24); }

struct LayerArgs {
    const __half* X;         // input tile images  [m_tiles][Kb][a_terms][8][128][8]
    const __half* W;         // weight tile images [2 terms][n_tiles][Kb][8][NT][8]
    const float* bias;       // [n_tiles * NT]
    __half* Y;               // next layer's X images [m_tiles][out_Kb][2][8][128][8], or null (last layer)
    float* logits; float* probs; float* values;      // last layer outputs (each may be null)
    int a_terms, Kb, NT, n_tiles, m_tiles, out_Kb, relu, num_actions, has_value, stages;
    long long batch;
    // dgrad (k_tc_layer<1>): Y = mask(X W) 2^(sexp[s_out] - sexp[s_in]); mask = the ReLU mask read from the images of the layer input,
    // [m_tiles][mask_Kb][2][8][128][8] (an entry is kept where its hi or lo half is non-zero)
    const __half* mask; const int* sexp; int s_in, s_out, mask_Kb;
};

struct SmemPlan { uint32_t a_off[kStages][2], b_off[kStages][2], bar_off, stage_off, total; };
// stages: pipeline depth of this layer (<= kStages); staging_floats: row-major [128][num_actions] output staging of the last layer (0 elsewhere)
__host__ __device__ inline SmemPlan plan_smem(int a_terms, int NT, int stages, int staging_floats) {
    SmemPlan p{}; uint32_t o = 0;
    for (int s = 0; s < stages; ++s) {
        for (int t = 0; t < 2; ++t) { p.a_off[s][t] = o; if (t < a_terms) o += kImgA * 2; }
        for (int t = 0; t < 2; ++t) { p.b_off[s][t] = o; o += (uint32_t)NT * kKB * 2; }
    }
    p.bar_off = o; o += 128;
    p.stage_off = o; o += (uint32_t)staging_floats * 4;
    p.total = o;
    return p;
}
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void epilogue_sync() { asm volatile("bar.sync 1, 128;\n" ::: "memory"); }      // the 4 epilogue warps

// kMode 0: the forward layer.  kMode 1: the dgrad of the backward pass (qg_policy_tc_backward): X = the layer's dZ images, W = its transposed
// weight images, the epilogue applies the ReLU mask of the layer's input and the power-of-two rescale instead of bias / ReLU
template <int kMode>
__global__ void __launch_bounds__(kThreads, 1) k_tc_layer(const __grid_constant__ LayerArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const SmemPlan sp = plan_smem(a.a_terms, a.NT, a.stages, a.Y ? 0 : kM * a.num_actions);
    const int kNumStages = a.stages;
    uint64_t* const full = reinterpret_cast<uint64_t*>(smem + sp.bar_off);      // [kStages]
    uint64_t* const empty = full + kStages;                                     // [kStages]
    uint64_t* const acc_full = empty + kStages;                                 // [2]
    float* const staging = reinterpret_cast<float*>(smem + sp.stage_off);
    uint64_t* const acc_empty = acc_full + 2;                                   // [2]
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = a.m_tiles * a.n_tiles;
    const uint32_t acc_cols = 128;                                              // columns per accumulator buffer (NT <= 128)

    if (threadIdx.x == 0) {
        for (int s = 0; s < kNumStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {            // one warp allocates the CTA's tensor memory: 2 accumulator buffers of 128 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(2 * acc_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // programmatic dependent launch: everything above overlapped the previous kernel of the stream; its results are needed from here on
    pdl_launch_dependents();
    pdl_wait();

    if (warp == 0) {
        // ===== loader =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            const uint32_t bytes = (uint32_t)a.a_terms * kImgA * 2 + 2u * (uint32_t)a.NT * kKB * 2;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int mt = t / a.n_tiles, nt = t - mt * a.n_tiles;
                for (int kb = 0; kb < a.Kb; ++kb) {
                    mbar_wait(empty + stage, phase ^ 1u);
                    mbar_expect_tx(full + stage, bytes);
                    for (int term = 0; term < a.a_terms; ++term)
                        bulk_g2s(smem + sp.a_off[stage][term], a.X + (((size_t)mt * a.Kb + kb) * a.a_terms + term) * kImgA, kImgA * 2, full + stage);
                    for (int term = 0; term < 2; ++term)
                        bulk_g2s(smem + sp.b_off[stage][term], a.W + (((size_t)term * a.n_tiles + nt) * a.Kb + kb) * ((size_t)a.NT * kKB), (uint32_t)a.NT * kKB * 2, full + stage);
                    if (++stage == (uint32_t)kNumStages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        {   // (the whole warp runs the issue loop, an elected lane issues: see umma_f16_w)
            uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
            const uint32_t idesc = instr_desc(a.NT);
            const uint32_t lbo_a = kM * 16, lbo_b = (uint32_t)a.NT * 16, sbo = 128;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                mbar_wait(acc_empty + as, aphase ^ 1u);             // the epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t d = tmem_base + as * acc_cols;
                for (int kb = 0; kb < a.Kb; ++kb) {
                    mbar_wait(full + stage, phase);
                    tc_fence_after();
                    const uint32_t sa0 = smem_u32(smem + sp.a_off[stage][0]), sa1 = smem_u32(smem + sp.a_off[stage][1]);
                    const uint32_t sb0 = smem_u32(smem + sp.b_off[stage][0]), sb1 = smem_u32(smem + sp.b_off[stage][1]);
#pragma unroll
                    for (int k = 0; k < kKB / 16; ++k) {            // one MMA covers K = 16: two 8-wide chunks, lbo apart
                        const uint64_t a_hi = smem_desc(sa0 + 2u * k * lbo_a, lbo_a, sbo), b_hi = smem_desc(sb0 + 2u * k * lbo_b, lbo_b, sbo);
                        const uint64_t b_lo = smem_desc(sb1 + 2u * k * lbo_b, lbo_b, sbo);
                        umma_f16_w(d, a_hi, b_hi, idesc, (kb | k) ? 1u : 0u);
                        umma_f16_w(d, a_hi, b_lo, idesc, 1u);
                        if (a.a_terms == 2) umma_f16_w(d, smem_desc(sa1 + 2u * k * lbo_a, lbo_a, sbo), b_hi, idesc, 1u);
                    }
                    umma_commit_w(empty + stage);                     // the stage is free once these MMAs have read it
                    if (++stage == (uint32_t)kNumStages) { stage = 0; phase ^= 1u; }
                }
                umma_commit_w(acc_full + as);                         // accumulator complete -> epilogue
                if (++as == 2) { as = 0; aphase ^= 1u; }
            }
        }
    } else {
        // ===== epilogue: warps 2..5; warp w may touch tensor-memory lanes 32 * (w % 4) .. + 31 =====
        const int q = warp & 3, row = q * 32 + lane;
        uint32_t as = 0, aphase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const int mt = t / a.n_tiles, nt = t - mt * a.n_tiles;
            mbar_wait(acc_full + as, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + as * acc_cols + ((uint32_t)(q * 32) << 16);
            const long long grow = (long long)mt * kM + row;
            if constexpr (kMode == 1) {
                const float f = ldexpf(1.0f, __ldg(a.sexp + a.s_out) - __ldg(a.sexp + a.s_in));
                for (int c0 = 0; c0 < a.NT; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(taddr + (uint32_t)c0, v);
                    const int n0 = nt * a.NT + c0;
                    const int okb = n0 >> 6, ch = (n0 & 63) >> 3;
                    const size_t at = ((size_t)ch * kM + row) * 8;
                    const __half* mimg = a.mask + (((size_t)mt * a.mask_Kb + okb) * 2) * kImgA;
                    const uint4* m_hi = reinterpret_cast<const uint4*>(mimg + at);
                    const uint4* m_lo = reinterpret_cast<const uint4*>(mimg + kImgA + at);
                    const uint4 h0 = m_hi[0], h1 = m_hi[kM], l0 = m_lo[0], l1 = m_lo[kM];
                    const uint32_t mw[8] = {h0.x | l0.x, h0.y | l0.y, h0.z | l0.z, h0.w | l0.w, h1.x | l1.x, h1.y | l1.y, h1.z | l1.z, h1.w | l1.w};
                    uint32_t hi[8], lo[8];
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        const float x0 = (mw[i >> 1] & 0xFFFFu) ? __uint_as_float(v[i]) * f : 0.0f;
                        const float x1 = (mw[i >> 1] >> 16) ? __uint_as_float(v[i + 1]) * f : 0.0f;
                        const __half hh0 = __float2half_rn(x0), hh1 = __float2half_rn(x1);
                        const __half ll0 = __float2half_rn(x0 - __half2float(hh0)), ll1 = __float2half_rn(x1 - __half2float(hh1));
                        hi[i >> 1] = (uint32_t)__half_as_ushort(hh0) | ((uint32_t)__half_as_ushort(hh1) << 16);
                        lo[i >> 1] = (uint32_t)__half_as_ushort(ll0) | ((uint32_t)__half_as_ushort(ll1) << 16);
                    }
                    __half* img = a.Y + (((size_t)mt * a.out_Kb + okb) * 2) * kImgA;
                    uint4* p_hi = reinterpret_cast<uint4*>(img + at);
                    uint4* p_lo = reinterpret_cast<uint4*>(img + kImgA + at);
                    p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]); p_hi[kM] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                    p_lo[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]); p_lo[kM] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
                }
            } else if (a.Y) {
                for (int c0 = 0; c0 < a.NT; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(taddr + (uint32_t)c0, v);
                    const int n0 = nt * a.NT + c0;
                    uint32_t hi[8], lo[8];
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        float x0 = __uint_as_float(v[i]) + __ldg(a.bias + n0 + i), x1 = __uint_as_float(v[i + 1]) + __ldg(a.bias + n0 + i + 1);
                        if (a.relu) { x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f); }
                        const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
                        const __half l0 = __float2half_rn(x0 - __half2float(h0)), l1 = __float2half_rn(x1 - __half2float(h1));
                        hi[i >> 1] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                        lo[i >> 1] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
                    }
                    // columns n0 .. n0+15 = K block n0 / 64 of the next layer, chunks (n0 % 64) / 8 and the one after
                    const int okb = n0 >> 6, ch = (n0 & 63) >> 3;
                    __half* img = a.Y + (((size_t)mt * a.out_Kb + okb) * 2) * kImgA;
                    uint4* p_hi = reinterpret_cast<uint4*>(img + ((size_t)ch * kM + row) * 8);
                    uint4* p_lo = reinterpret_cast<uint4*>(img + kImgA + ((size_t)ch * kM + row) * 8);
                    p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]); p_hi[kM] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                    p_lo[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]); p_lo[kM] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
                }
            } else {
                // last layer: columns 0 .. A-1 are the action logits, column A the value head.  The row's logits are read from tensor memory once
                // into registers (fully unrolled: NT <= 128), soft-maxed there, and leave through a row-major staging tile in shared memory so
                // that the tile's [128][A] block of the output — contiguous in the [B][A] tensor — is written with coalesced stores
                const int A = a.num_actions;
                float x[kMaxNT];
#pragma unroll
                for (int c = 0; c < kMaxNT / 16; ++c) {
                    if (c * 16 < a.NT) {
                        uint32_t v[16];
                        tmem_ld16(taddr + (uint32_t)(c * 16), v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) x[c * 16 + i] = __uint_as_float(v[i]) + __ldg(a.bias + c * 16 + i);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty + as);         // the accumulator is in registers: the MMA warp may reuse the buffer now
                if (a.has_value && a.values && grow < a.batch) {
                    float val = 0.0f;
#pragma unroll
                    for (int n = 0; n < kMaxNT; ++n) if (n == A) val = x[n];
                    a.values[grow] = val;
                }
                const long long rows_left = a.batch - (long long)mt * kM;
                const int nrows = rows_left < kM ? (int)rows_left : kM;
                float* const srow = staging + (size_t)row * A;
                auto flush = [&](float* out) {                       // staging [nrows][A] -> out rows mt*128 .., coalesced
                    epilogue_sync();
                    float* dst = out + (size_t)mt * kM * A;
                    const int tid = row, total = nrows * A;
                    for (int i = tid; i < total; i += 128) dst[i] = staging[i];
                    epilogue_sync();
                };
                if (a.logits) {
#pragma unroll
                    for (int n = 0; n < kMaxNT; ++n) if (n < A) srow[n] = x[n];
                    flush(a.logits);
                }
                if (a.probs) {
                    float mx = -INFINITY, sum = 0.0f;
#pragma unroll
                    for (int n = 0; n < kMaxNT; ++n) if (n < A) mx = fmaxf(mx, x[n]);
#pragma unroll
                    for (int n = 0; n < kMaxNT; ++n) if (n < A) { x[n] = expf(x[n] - mx); sum += x[n]; }
                    const float inv = 1.0f / sum;
#pragma unroll
                    for (int n = 0; n < kMaxNT; ++n) if (n < A) srow[n] = x[n] * inv;
                    flush(a.probs);
                }
                if (++as == 2) { as = 0; aphase ^= 1u; }
                continue;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + as);             // 4 epilogue warps -> buffer free for the MMA warp
            if (++as == 2) { as = 0; aphase ^= 1u; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(2 * acc_cols) : "memory");
}

// ---- the three layers of a BasicPolicy (embeddings -> one common layer -> action / value head) in ONE kernel ------------------------------
// The per-layer kernels above push every hidden activation through global memory twice (h1: 2 x 134 MB at 65 536 rows).  Here a CTA keeps its
// 128 rows on chip from the observation tile to the logits:
//   layer 1 is computed in 128-column chunks (accumulators D1[0] / D1[1] in tensor memory, double buffered); the epilogue turns a finished
//   chunk into f16 hi/lo halves in a 64 KB shared-memory buffer laid out as TWO K blocks of layer 2's A operand; layer 2 accumulates those two
//   K blocks into D2 (256 columns) while layer 1's next chunk is already being multiplied; when the last chunk is in, D2 is turned — 128 columns
//   at a time, through the same buffer — into layer 3's A operand, and the head's accumulator takes the place of a D1 buffer.
// Tensor memory: D1[0] cols 0..127, D1[1] cols 128..255, D2 cols 256..511.  Shared memory: 2 ring stages of 64 KB (weight tiles, and layer
// 1's observation tiles) + the 64 KB activation buffer (which doubles as the output staging tile of the head).
//   warp 0 loader, warp 1 MMA issuer (the whole warp runs the issue loop, an elected lane issues: umma_f16_lo), warps 2..9 epilogue (two warps
//   per tensor-memory lane quarter, each converting half of the columns; all eight share the head's soft-max), warps 10..13 expand the packed
//   observation bits of the CTA's 128 rows (one row per thread, words requested one stage ahead) into layer 1's A tile of every layer-1 stage
//   (0 / 1 as f16: one 16-byte store per 8 entries) — no expansion pre-pass, no A tiles in global memory, a fifth less traffic into shared memory.
// Where the time goes (tools build -DQG_TC_PROBE, profiles/r2_v42_tc_probe.json; 65 536 rows = 512 tiles on 148 CTAs): the MMA-issuing thread
// waits 9 % for layer 2's activation halves, 6 % each for layer 1's weights and observation tiles, 6 % for the head's input, 3 % for a free
// accumulator; a CTA with 4 tiles sets the kernel's time while the mean is 3.46 (wave quantisation: 13 %).  Tried and measured slower: four
// 32 KB half-K-block ring stages (126 vs 122 us), two activation buffers + three stages (138 us), a shared-memory byte table for the producers
// (114 vs 100 us: its loads compete with the operand reads), converting a chunk into registers before its buffer is free (spills).
struct FusedArgs {
    const uint32_t* bits;    // packed observations [batch][obs_words]: layer 1's A tiles are expanded from them inside the kernel
    int obs_words, obs_size;
    const __half* X0;        // (unused by the fused kernel: observation tile images of the per-layer path)
    const __half* W1;        // [2 terms][NC chunks][Kb0][8][128][8]
    const __half* W2;        // [2 terms][Kb2 = E_pad / 64][8][C_pad][8]
    const __half* W3;        // [2 terms][Kb3 = C_pad / 64][8][H][8]
    const float* b1; const float* b2; const float* b3;
    float* logits; float* probs; float* values;
    int Kb0, NC, C_pad, Kb3, H, m_tiles, num_actions, has_value;
    long long batch;
};
constexpr int kProducerWarps = 4;         // observation-tile producers: one row per thread
constexpr int kFusedThreads = 320 + 32 * kProducerWarps;        // loader, MMA, 8 epilogue warps, the producers
constexpr uint32_t kRingStage = 64 * 1024, kActBytes = 64 * 1024;
constexpr uint32_t kFusedBias = (512 + 256 + 128) * 4;        // the three bias vectors, staged once per CTA (NC <= 4, C_pad <= 256, H <= 128)
constexpr uint32_t kFusedRed = 4 * 128 * 4;                   // the head's partial row maxima / sums of the two warps of a lane quarter
constexpr uint32_t kFusedSmem = 2 * kRingStage + kActBytes + 256 + kFusedBias + kFusedRed;
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void epilogue8_sync() { asm volatile("bar.sync 2, 256;\n" ::: "memory"); }
__device__ __forceinline__ void epilogue4_sync() { asm volatile("bar.sync 3, 128;\n" ::: "memory"); }

__global__ void __launch_bounds__(kFusedThreads, 1) k_tc_fused3(const __grid_constant__ FusedArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* const ring = smem;                         // [2][64 KB]
    uint8_t* const act = smem + 2 * kRingStage;         // hi: K blocks 0, 1 (16 KB each) | lo: K blocks 0, 1
    uint64_t* const bars = reinterpret_cast<uint64_t*>(act + kActBytes);
    uint64_t* const full = bars;            // [2]
    uint64_t* const empty = bars + 2;       // [2]
    uint64_t* const d1_full = bars + 4;     // [2]
    uint64_t* const d1_empty = bars + 6;    // [2]
    uint64_t* const d2_full = bars + 8;
    uint64_t* const d2_empty = bars + 9;
    uint64_t* const act_full = bars + 10;   // [2]: one pair of barriers per K block of the activation buffer (columns 0..63 / 64..127 of a
    uint64_t* const act_empty = bars + 12;  // [2]  128-column piece): the epilogue refills K block 0 while the products of K block 1 still run
    uint64_t* const a0_full = bars + 14;    // [2]: the producers' part of a layer-1 stage (the observation tile) is written
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
    float* const sb1 = reinterpret_cast<float*>(act + kActBytes + 256);       // biases in shared memory: the epilogue reads them with broadcast
    float* const sb2 = sb1 + 512;                                              // 16-byte loads instead of one global load per column (those
    float* const sb3 = sb2 + 256;                                              // were the epilogue's top stall: long_scoreboard, ncu r2_v11)
    float* const red_max = sb3 + 128;                                          // [2][128]
    float* const red_sum = red_max + 2 * kM;                                   // [2][128]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int halves = (a.C_pad + 127) / 128;           // D2 leaves in 128-column pieces

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); mbar_init(d1_full + s, 1); mbar_init(d1_empty + s, 8); }
        mbar_init(d2_full, 1); mbar_init(d2_empty, 8);
        for (int j = 0; j < 2; ++j) { mbar_init(act_full + j, 4); mbar_init(act_empty + j, 1); mbar_init(a0_full + j, kProducerWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_launch_dependents();
    pdl_wait();
    for (int i = threadIdx.x; i < a.NC * 128; i += kFusedThreads) sb1[i] = a.b1[i];
    for (int i = threadIdx.x; i < a.C_pad; i += kFusedThreads) sb2[i] = a.b2[i];
    for (int i = threadIdx.x; i < a.H; i += kFusedThreads) sb3[i] = a.b3[i];
    __syncthreads();

    const uint32_t img128 = 128 * kKB;                  // halves per 128-row K-block image
    if (warp == 0) {
        // ===== loader: the stages in the order the MMA warp consumes them =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            auto next = [&]() { if (++stage == 2) { stage = 0; phase ^= 1u; } };
            auto stage_l1 = [&](int mt, int c, int kb) {
                mbar_wait(empty + stage, phase ^ 1u);
                uint8_t* sp = ring + stage * kRingStage;
                mbar_expect_tx(full + stage, 2u * img128 * 2);           // (the first 16 KB of the stage is the producers' observation tile)
                bulk_g2s(sp + 16384, a.W1 + (((size_t)0 * a.NC + c) * a.Kb0 + kb) * img128, img128 * 2, full + stage);
                bulk_g2s(sp + 32768, a.W1 + (((size_t)1 * a.NC + c) * a.Kb0 + kb) * img128, img128 * 2, full + stage);
                next();
            };
            auto stage_w = [&](const __half* W, int kbs, int rows, int kb) {       // hi at +0, lo at +32 KB
                mbar_wait(empty + stage, phase ^ 1u);
                uint8_t* sp = ring + stage * kRingStage;
                const uint32_t bytes = (uint32_t)rows * kKB * 2;
                mbar_expect_tx(full + stage, 2u * bytes);
                bulk_g2s(sp, W + ((size_t)0 * kbs + kb) * ((size_t)rows * kKB), bytes, full + stage);
                bulk_g2s(sp + 32768, W + ((size_t)1 * kbs + kb) * ((size_t)rows * kKB), bytes, full + stage);
                next();
            };
            for (int mt = blockIdx.x; mt < a.m_tiles; mt += gridDim.x) {
                for (int c = 0; c <= a.NC; ++c) {
                    if (c < a.NC) for (int kb = 0; kb < a.Kb0; ++kb) stage_l1(mt, c, kb);
                    if (c > 0) for (int j = 0; j < 2; ++j) stage_w(a.W2, 2 * a.NC, a.C_pad, 2 * (c - 1) + j);
                }
                for (int kb = 0; kb < a.Kb3; ++kb) stage_w(a.W3, a.Kb3, a.H, kb);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        {   // (the whole warp: see umma_f16_w)
            uint32_t stage = 0, phase = 0;
#ifdef QG_TC_PROBE
            long long tcw[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const long long tc_t0 = clock64();
#endif
            uint32_t n_d1e[2] = {0, 0}, n_actf[2] = {0, 0}, n_d2e = 0, n_a0[2] = {0, 0};  // waits done so far on d1_empty[b], act_full[j], d2_empty, a0_full[s]
            const uint32_t lbo128 = 128 * 16;
            const uint32_t id1 = instr_desc(128), id2 = instr_desc(a.C_pad), id3 = instr_desc(a.H);
            const uint32_t lbo2 = (uint32_t)a.C_pad * 16, lbo3 = (uint32_t)a.H * 16;
            const uint32_t ks128 = 2u * lbo128 >> 4, ks2 = 2u * lbo2 >> 4, ks3 = 2u * lbo3 >> 4;    // descriptor step per K = 16 slice (two 8-wide k groups)
            const uint32_t act_u = smem_u32(act);
            auto next = [&]() { if (++stage == 2) { stage = 0; phase ^= 1u; } };
            for (int mt = blockIdx.x; mt < a.m_tiles; mt += gridDim.x) {
                for (int c = 0; c <= a.NC; ++c) {
                    if (c < a.NC) {
                        // layer 1, chunk c -> D1[c & 1]
                        const int b = c & 1;
                        TC_MMA_WAIT(0, d1_empty + b, (n_d1e[b] & 1u) ^ 1u); ++n_d1e[b];
                        tc_fence_after();
                        const uint32_t d = tmem_base + (uint32_t)b * 128;
                        for (int kb = 0; kb < a.Kb0; ++kb) {
                            TC_MMA_WAIT(1, full + stage, phase);
                            TC_MMA_WAIT(2, a0_full + stage, n_a0[stage] & 1u); ++n_a0[stage];
                            tc_fence_after();
                            const uint32_t sp = smem_u32(ring + stage * kRingStage);
                            const uint32_t a0 = desc_lo(sp, lbo128), b0 = desc_lo(sp + 16384, lbo128), b1 = desc_lo(sp + 32768, lbo128);
#pragma unroll
                            for (int k = 0; k < kKB / 16; ++k) {
                                umma_f16_lo(d, a0 + k * ks128, b0 + k * ks128, id1, (kb | k) ? 1u : 0u);
                                umma_f16_lo(d, a0 + k * ks128, b1 + k * ks128, id1, 1u);
                            }
                            umma_commit_w(empty + stage);
                            next();
                        }
                        umma_commit_w(d1_full + b);
                    }
                    if (c > 0) {
                        // layer 2 over the two K blocks of chunk c - 1 (the epilogue's halves in the activation buffer) -> D2
                        if (c == 1) { TC_MMA_WAIT(3, d2_empty, (n_d2e & 1u) ^ 1u); ++n_d2e; }
                        const uint32_t d = tmem_base + 256;
                        for (int j = 0; j < 2; ++j) {
                            TC_MMA_WAIT(4, act_full + j, n_actf[j] & 1u); ++n_actf[j];
                            TC_MMA_WAIT(5, full + stage, phase);
                            tc_fence_after();
                            const uint32_t sp = smem_u32(ring + stage * kRingStage);
                            const uint32_t a_hi = act_u + (uint32_t)j * 16384, a_lo = act_u + 32768 + (uint32_t)j * 16384;
                            const uint32_t ah0 = desc_lo(a_hi, lbo128), al0 = desc_lo(a_lo, lbo128), bh0 = desc_lo(sp, lbo2), bl0 = desc_lo(sp + 32768, lbo2);
#pragma unroll
                            for (int k = 0; k < kKB / 16; ++k) {
                                umma_f16_lo(d, ah0 + k * ks128, bh0 + k * ks2, id2, (c > 1 || j || k) ? 1u : 0u);
                                umma_f16_lo(d, ah0 + k * ks128, bl0 + k * ks2, id2, 1u);
                                umma_f16_lo(d, al0 + k * ks128, bh0 + k * ks2, id2, 1u);
                            }
                            umma_commit_w(empty + stage);
                            umma_commit_w(act_empty + j);              // this K block may be rewritten once these products have read it
                            next();
                        }
                    }
                }
                umma_commit_w(d2_full);
                // the head: layer 3 over the halves of D2 as they come back through the activation buffer -> the D1 buffer whose turn it is
                {
                    const int b = a.NC & 1;
                    TC_MMA_WAIT(0, d1_empty + b, (n_d1e[b] & 1u) ^ 1u); ++n_d1e[b];
                    tc_fence_after();
                    const uint32_t d = tmem_base + (uint32_t)b * 128;
                    for (int h = 0; h < halves; ++h) {
                        const int kbs = min(2, a.Kb3 - 2 * h);
                        for (int j = 0; j < kbs; ++j) {
                            TC_MMA_WAIT(6, act_full + j, n_actf[j] & 1u); ++n_actf[j];
                            TC_MMA_WAIT(5, full + stage, phase);
                            tc_fence_after();
                            const uint32_t sp = smem_u32(ring + stage * kRingStage);
                            const uint32_t a_hi = act_u + (uint32_t)j * 16384, a_lo = act_u + 32768 + (uint32_t)j * 16384;
                            const uint32_t ah0 = desc_lo(a_hi, lbo128), al0 = desc_lo(a_lo, lbo128), bh0 = desc_lo(sp, lbo3), bl0 = desc_lo(sp + 32768, lbo3);
#pragma unroll
                            for (int k = 0; k < kKB / 16; ++k) {
                                umma_f16_lo(d, ah0 + k * ks128, bh0 + k * ks3, id3, (h || j || k) ? 1u : 0u);
                                umma_f16_lo(d, ah0 + k * ks128, bl0 + k * ks3, id3, 1u);
                                umma_f16_lo(d, al0 + k * ks128, bh0 + k * ks3, id3, 1u);
                            }
                            umma_commit_w(empty + stage);
                            umma_commit_w(act_empty + j);
                            next();
                        }
                    }
                    umma_commit_w(d1_full + b);
                }
            }
#ifdef QG_TC_PROBE
            tcw[7] = clock64() - tc_t0;
            if (lane == 0 && blockIdx.x < 160) for (int i = 0; i < 8; ++i) g_tc_wait[blockIdx.x * 8 + i] = tcw[i];
#endif
        }
    } else if (warp >= 10) {
        // ===== observation-tile producers: follow the loader's stage sequence; for every layer-1 stage write rows' 64 entries of K block kb =====
        const int row = threadIdx.x - 320;               // 0..127
        uint32_t stage = 0, phase = 0;
        auto next = [&]() { if (++stage == 2) { stage = 0; phase ^= 1u; } };
        // the two observation words of K block kb of this thread's row, masked to the entries that exist.  They are requested one stage ahead:
        // a stage's turn-around (stage free -> tile written) then holds no global-memory latency
        auto load_words = [&](int mt, int kb, uint32_t (&w)[2]) {
            const long long grow = (long long)mt * kM + row;
            uint32_t w0 = 0, w1 = 0;
            if (grow < a.batch) {
                const uint32_t* src = a.bits + (size_t)grow * a.obs_words;
                if (2 * kb < a.obs_words) w0 = __ldg(src + 2 * kb);
                if (2 * kb + 1 < a.obs_words) w1 = __ldg(src + 2 * kb + 1);
                const int left = a.obs_size - kb * 64;           // entries of this K block that exist
                if (left < 32) w0 &= left > 0 ? ((1u << left) - 1u) : 0u;
                if (left < 64) w1 &= left > 32 ? ((1u << (left - 32)) - 1u) : 0u;
            }
            w[0] = w0; w[1] = w1;
        };
        for (int mt = blockIdx.x; mt < a.m_tiles; mt += gridDim.x) {
            uint32_t wn[2];
            load_words(mt, 0, wn);
            for (int c = 0; c <= a.NC; ++c) {
                if (c < a.NC) {
                    for (int kb = 0; kb < a.Kb0; ++kb) {
                        const uint32_t wc[2] = {wn[0], wn[1]};
                        load_words(mt, kb + 1 < a.Kb0 ? kb + 1 : 0, wn);          // (the next chunk starts over at K block 0)
                        mbar_wait(empty + stage, phase ^ 1u);            // the products that read this stage's previous contents are done
                        uint8_t* const tile = ring + stage * kRingStage;
#pragma unroll
                        for (int ch = 0; ch < 8; ++ch) {
                            // 8 entries as f16 0 / 1.  (A 256-entry shared-memory table instead of these selects was measured: 114 instead of
                            // 100 us per forward — its loads compete with the tensor core's operand reads for the shared-memory bandwidth.)
                            const uint32_t b = (wc[ch >> 2] >> ((ch & 3) * 8)) & 0xFFu;
                            uint4 o;
                            o.x = ((b & 1u) ? 0x3C00u : 0u) | ((b & 2u) ? 0x3C000000u : 0u);
                            o.y = ((b & 4u) ? 0x3C00u : 0u) | ((b & 8u) ? 0x3C000000u : 0u);
                            o.z = ((b & 16u) ? 0x3C00u : 0u) | ((b & 32u) ? 0x3C000000u : 0u);
                            o.w = ((b & 64u) ? 0x3C00u : 0u) | ((b & 128u) ? 0x3C000000u : 0u);
                            *reinterpret_cast<uint4*>(tile + ((size_t)ch * kM + row) * 16) = o;
                        }
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(a0_full + stage);
                        next();
                    }
                }
                // layer 2's two weight stages are not the producers' business, but every use of a stage has to be waited for: a parity
                // wait can only tell the phase it expects from the one before it, so a waiter must never fall two phases behind
                if (c > 0) for (int j = 0; j < 2; ++j) { mbar_wait(empty + stage, phase ^ 1u); next(); }
            }
            for (int kb = 0; kb < a.Kb3; ++kb) { mbar_wait(empty + stage, phase ^ 1u); next(); }      // the head's weight stages
        }
    } else {
        // ===== epilogue: warps 2..9.  Quarter q = warp % 4 owns tensor-memory lanes 32q..32q+31 (rows); of the two warps of a quarter the one
        // with hsel = 0 converts columns 0..63 of a 128-column piece (K block 0 of the buffer), the other columns 64..127 (K block 1) =====
        const int q = warp & 3, hsel = (warp - 2) >> 2, row = q * 32 + lane;
        uint32_t n_d1f[2] = {0, 0}, n_acte = 0, n_d2f = 0;
#ifdef QG_TC_PROBE
        long long tce[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const long long tce_t0 = clock64();
#endif
        const uint32_t lane_base = ((uint32_t)(q * 32) << 16);
        // 64 accumulator columns starting at tensor-memory column `tcol` -> + bias, ReLU, hi / lo halves -> K block `hsel` of the buffer.
        // (Tried: converting into 64 registers before waiting for act_empty, so that only the shared-memory stores sit between act_empty
        // and act_full — 158 instead of 133 us per 65 536-row forward: the longer live ranges spill, profiles/r2_v12_tc_probe.json.)
        auto convert64 = [&](uint32_t tcol, const float* bias) {
            uint8_t* const kb_hi = act + (uint32_t)hsel * 16384;
            uint8_t* const kb_lo = kb_hi + 32768;
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(tmem_base + lane_base + tcol + (uint32_t)c0, v);
                uint32_t hi[8], lo[8];
                float bb[16];
#pragma unroll
                for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(bb + i) = *reinterpret_cast<const float4*>(bias + c0 + i);
#pragma unroll
                for (int i = 0; i < 16; i += 2) {
                    const float x0 = fmaxf(__uint_as_float(v[i]) + bb[i], 0.0f), x1 = fmaxf(__uint_as_float(v[i + 1]) + bb[i + 1], 0.0f);
                    const __half2 h2 = __floats2half2_rn(x0, x1);
                    const float2 hf = __half22float2(h2);
                    const __half2 l2 = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                    hi[i >> 1] = *reinterpret_cast<const uint32_t*>(&h2);
                    lo[i >> 1] = *reinterpret_cast<const uint32_t*>(&l2);
                }
                const int ch = c0 >> 3;                               // 8-column chunk within the K block
                uint4* p_hi = reinterpret_cast<uint4*>(kb_hi + ((size_t)ch * kM + row) * 16);
                uint4* p_lo = reinterpret_cast<uint4*>(kb_lo + ((size_t)ch * kM + row) * 16);
                p_hi[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]); p_hi[kM] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                p_lo[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]); p_lo[kM] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
            }
        };
        auto publish = [&]() {                                        // this warp's part of the buffer is written: hand it to the tensor core
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(act_full + hsel);
        };
        for (int mt = blockIdx.x; mt < a.m_tiles; mt += gridDim.x) {
            for (int c = 0; c < a.NC; ++c) {
                const int b = c & 1;
                TC_EPI(0, mbar_wait(d1_full + b, n_d1f[b] & 1u)); ++n_d1f[b];
                TC_EPI(1, mbar_wait(act_empty + hsel, (n_acte & 1u) ^ 1u)); ++n_acte;   // the previous chunk's layer-2 products have read this K block
                tc_fence_after();
                TC_EPI(2, convert64((uint32_t)b * 128 + (uint32_t)hsel * 64, sb1 + c * 128 + hsel * 64);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(d1_empty + b);
                publish());
            }
            TC_EPI(3, mbar_wait(d2_full, n_d2f & 1u)); ++n_d2f;
#ifdef QG_TC_PROBE
            const long long tce_t4 = clock64();
#endif
            for (int h = 0; h < halves; ++h) {
                const bool mine = h * 128 + hsel * 64 < a.C_pad;       // (a K block past C_pad does not exist: the MMA warp does not wait for it)
                if (mine) { mbar_wait(act_empty + hsel, (n_acte & 1u) ^ 1u); ++n_acte; }
                tc_fence_after();
                if (mine) convert64(256u + (uint32_t)h * 128 + (uint32_t)hsel * 64, sb2 + h * 128 + hsel * 64);
                if (h == halves - 1) { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(d2_empty); }
                if (mine) publish();
            }
#ifdef QG_TC_PROBE
            tce[4] += clock64() - tce_t4;
            const long long tce_t6 = clock64();
#endif
            // the head's accumulator.  All 8 epilogue warps share it: of the two warps of a tensor-memory lane quarter the one with hsel = 0 takes
            // the head's columns below `split`, the other the rest (measured with four warps holding whole rows — 128 live registers per thread,
            // a 128-entry predicated soft-max loop, 8-way bank conflicts on a row stride of A floats: 17 us of a tile's 30, the MMA thread idle
            // behind it; profiles/r2_v34_tc_probe.json).  The pair's partial maxima / sums meet in shared memory; the staging tile has an odd
            // row stride and leaves row by row, coalesced.
            {
                const int b = a.NC & 1;
                TC_EPI(5, mbar_wait(d1_full + b, n_d1f[b] & 1u)); ++n_d1f[b];
                tc_fence_after();
                const int A = a.num_actions;
                const long long grow = (long long)mt * kM + row;
                const int split = ((a.H + 31) / 32) * 16;             // a multiple of 16 (tcgen05.ld width), <= 64
                const int col0 = hsel ? split : 0, ncols = hsel ? a.H - split : split;
                float x[64];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c * 16 < ncols) {
                        uint32_t v[16];
                        tmem_ld16(tmem_base + lane_base + (uint32_t)b * 128 + (uint32_t)(col0 + c * 16), v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) x[c * 16 + i] = __uint_as_float(v[i]) + sb3[col0 + c * 16 + i];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(d1_empty + b);             // (all 8 warps arrive: the barrier's count is the same for every use)
                const int na = min(max(A - col0, 0), ncols);          // this warp's action columns: x[0 .. na)
                if (a.has_value && a.values && grow < a.batch && A >= col0 && A < col0 + ncols) {
                    float val = 0.0f;
#pragma unroll
                    for (int n = 0; n < 64; ++n) if (n == A - col0) val = x[n];
                    a.values[grow] = val;
                }
                // the activation buffer is idle until the next tile's first chunk (these same warps write it): it is the staging tile
                float* const staging = reinterpret_cast<float*>(act);
                // row stride of the staging tile: A % 4 == 0 -> 4 (mod 8) floats, so that the 16-byte stores of the 8 lanes of a quarter-warp
                // (8 rows) cover all 32 banks, and rows leave as float4; otherwise odd, scalar stores
                const bool vec = (A & 3) == 0;
                const int SA = vec ? A + ((12 - (A & 7)) & 7) : (A | 1);
                const long long rows_left = a.batch - (long long)mt * kM;
                const int nrows = rows_left < kM ? (int)rows_left : kM;
                float* const srow = staging + (size_t)row * SA + col0;
                const int et = threadIdx.x - 64;                      // 0..255 over the 8 epilogue warps
                auto stage_row = [&](float scale) {
                    if (vec) {
#pragma unroll
                        for (int n = 0; n < 64; n += 4) if (n < na) *reinterpret_cast<float4*>(srow + n) = make_float4(x[n] * scale, x[n + 1] * scale, x[n + 2] * scale, x[n + 3] * scale);
                    } else {
#pragma unroll
                        for (int n = 0; n < 64; ++n) if (n < na) srow[n] = x[n] * scale;
                    }
                };
                auto flush = [&](float* out) {                        // staging [nrows][SA] -> out rows mt * 128 .. (contiguous: row stride A), coalesced
                    epilogue8_sync();
                    float* dst = out + (size_t)mt * kM * A;
                    if (vec) {
                        const int a4 = A >> 2, total = nrows * a4;
                        for (int i = et; i < total; i += 256) {
                            const int r = i / a4, c4 = i - r * a4;
                            reinterpret_cast<float4*>(dst)[i] = *reinterpret_cast<const float4*>(staging + (size_t)r * SA + 4 * c4);
                        }
                    } else {
                        for (int r = et >> 5; r < nrows; r += 8) for (int cc = lane; cc < A; cc += 32) dst[(size_t)r * A + cc] = staging[(size_t)r * SA + cc];
                    }
                    epilogue8_sync();
                };
                // A % 4 == 0: every thread writes its columns of its row straight from registers as float4 (a row is A contiguous floats; the 32
                // rows of a warp make 32 half-used sectors per store, which L2 merges) — staging tile, two block barriers and the copy loop cost
                // more than the uncoalesced stores (profiles/r2_v40_tc_probe.json -> r2_v41)
                auto store_row = [&](float* out, float scale) {
                    if (grow < a.batch) {
                        float* drow = out + (size_t)grow * A + col0;
#pragma unroll
                        for (int n = 0; n < 64; n += 4) if (n < na) *reinterpret_cast<float4*>(drow + n) = make_float4(x[n] * scale, x[n + 1] * scale, x[n + 2] * scale, x[n + 3] * scale);
                    }
                };
                if (a.logits) {
                    if (vec) store_row(a.logits, 1.0f);
                    else { stage_row(1.0f); flush(a.logits); }
                }
                if (a.probs) {
                    float mx = -INFINITY, sum = 0.0f;
#pragma unroll
                    for (int n = 0; n < 64; ++n) if (n < na) mx = fmaxf(mx, x[n]);
                    red_max[hsel * kM + row] = mx;
                    epilogue8_sync();
                    mx = fmaxf(red_max[row], red_max[kM + row]);
#pragma unroll
#ifdef QG_TC_FASTEXP         // (tools A/B build: ex2.approx instead of the full-precision expf)
                    for (int n = 0; n < 64; ++n) if (n < na) { x[n] = __expf(x[n] - mx); sum += x[n]; }
#else
                    for (int n = 0; n < 64; ++n) if (n < na) { x[n] = expf(x[n] - mx); sum += x[n]; }
#endif
                    red_sum[hsel * kM + row] = sum;
                    epilogue8_sync();
                    const float inv = 1.0f / (red_sum[row] + red_sum[kM + row]);
                    if (vec) store_row(a.probs, inv);
                    else { stage_row(inv); flush(a.probs); }
                }
                if (!vec) epilogue8_sync();      // (no warp starts the next tile's first chunk in the buffer while it is the staging tile)
            }
#ifdef QG_TC_PROBE
            tce[6] += clock64() - tce_t6;
#endif
        }
#ifdef QG_TC_PROBE
        tce[7] = clock64() - tce_t0;
        if (warp == 2 && lane == 0 && blockIdx.x < 160) for (int i = 0; i < 8; ++i) g_tc_epi[blockIdx.x * 8 + i] = tce[i];
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512) : "memory");
}

// packed observation bits -> the first layer's X tile images (one half per entry: 0 / 1 are exact): thread = (row, 8-column chunk)
__global__ void k_tc_expand_bits(const uint32_t* __restrict__ bits, int obs_words, int obs_size, long long batch, int Kb, __half* __restrict__ X, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int row = (int)(i % kM);
    long long r = i / kM;
    const int ch = (int)(r % 8); r /= 8;
    const int kb = (int)(r % Kb);
    const long long mt = r / Kb;
    const long long grow = mt * kM + row;
    const int col0 = kb * kKB + ch * 8;
    uint32_t b = 0;
    if (grow < batch && col0 < obs_size) {
        b = (bits[(size_t)grow * obs_words + (col0 >> 5)] >> (col0 & 31)) & 0xFFu;
        if (col0 + 8 > obs_size) b &= (1u << (obs_size - col0)) - 1u;
    }
    const uint32_t one = 0x3C00u;     // half(1.0)
    uint4 o;
    o.x = ((b & 1u) ? one : 0u) | ((b & 2u) ? one << 16 : 0u);
    o.y = ((b & 4u) ? one : 0u) | ((b & 8u) ? one << 16 : 0u);
    o.z = ((b & 16u) ? one : 0u) | ((b & 32u) ? one << 16 : 0u);
    o.w = ((b & 64u) ? one : 0u) | ((b & 128u) ? one << 16 : 0u);
    reinterpret_cast<uint4*>(X)[i] = o;       // image order [mt][kb][ch][row] x 16 bytes == i
}

// in-place weight refresh (qg_policy_tc_load_weights_dev): f32 weights [rows][K] (row `rows` = the value head's when vw is set) -> the
// [term][n_tile][kb][k/8][n][k%8] hi / lo images qg_policy_tc_create lays out on the host, same split; bias[n] alongside (when bias is set).
// Padding rows / columns are not touched: they stay the zeros of creation.  Thread = (row, k), so the f32 rows are read coalesced
__global__ void k_tc_load_layer(const float* __restrict__ W, const float* __restrict__ b, const float* __restrict__ vw, const float* __restrict__ vb,
                                int rows, int K, int NT, int n_tiles, int Kb, __half* __restrict__ img, float* __restrict__ bias) {
    const int nrows = rows + (vw ? 1 : 0);
    const long long total = (long long)nrows * K, term = (long long)n_tiles * Kb * NT * kKB;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i / K), k = (int)(i - (long long)n * K);
        const bool vrow = n == rows;
        const float w = vrow ? vw[k] : W[i];
        const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
        const int nt = n / NT, nl = n - nt * NT, kb = k / kKB, kl = k - kb * kKB;
        const long long at = ((long long)nt * Kb + kb) * NT * kKB + ((long long)(kl >> 3) * NT + nl) * 8 + (kl & 7);
        img[at] = hi;
        img[term + at] = lo;
        if (bias && k == 0) bias[n] = vrow ? *vb : b[n];
    }
}

// ---- the backward pass (qg_policy_tc_backward) ----------------------------------------------------------------------------------------------
// dZ of every layer is carried like an activation: hi / lo images [m_tiles][KbZ][2][8][128][8], KbZ even (wgrad reads 128 columns per tile),
// scaled by 2^sexp[l] so that the halves of PPO's ~1e-6 mean-loss gradients are not f16 subnormals.  sexp comes from a device-side amax of the
// head's gradient and, layer by layer, from the bound max|dZ_(l-1)| <= max|dZ_l| colsum_l (colsum_l = max_k sum_n |W_l[n][k]|, computed when
// the weights are loaded): every scaled value stays below 2^15, no host synchronisation, no second pass.
constexpr int kChunkTiles = 8;       // wgrad's split-K chunk: 8 row tiles = 1024 rows, whatever the handle's capacity or the SM count

__device__ __forceinline__ uint32_t f32_abs_bits(float x) { return __float_as_uint(x) & 0x7FFFFFFFu; }
__device__ __forceinline__ int scale_exp(float b) {        // the largest s with b 2^s < 2^15 (0 for a zero or non-finite bound)
    if (!(b > 0.0f) || !isfinite(b)) return 0;
    int e; frexpf(b, &e);                                   // b < 2^e
    return max(-100, min(100, 15 - e));
}
__device__ __forceinline__ void atomic_max_bits(uint32_t* dst, uint32_t v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    if ((threadIdx.x & 31) == 0 && v) atomicMax(dst, v);
}
// amax[0] = max |dlogits|, |dvalues| (as f32 bits: non-negative floats order like their bits; a NaN compares above +inf)
__global__ void k_tc_amax(const float* __restrict__ dl, long long n_dl, const float* __restrict__ dv, long long n_dv, uint32_t* amax) {
    uint32_t m = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_dl + n_dv; i += (long long)gridDim.x * blockDim.x)
        m = max(m, f32_abs_bits(i < n_dl ? dl[i] : dv[i - n_dl]));
    atomic_max_bits(amax, m);
}
// colsum[l] (as f32 bits) = max over input columns k of sum_n |hi + lo| of the layer's forward weight images, inflated by 2^-9 (hi + lo is w to
// 2^-22; the bound must not be below the true one)
__global__ void k_tc_colsum(const __half* __restrict__ img, int N, int K, int NT, int n_tiles, int Kb, uint32_t* out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    float s = 0.0f;
    if (k < K) {
        const long long term = (long long)n_tiles * Kb * NT * kKB;
        const int kb = k / kKB, kl = k - kb * kKB;
        for (int n = 0; n < N; ++n) {
            const int nt = n / NT, nl = n - nt * NT;
            const long long at = ((long long)nt * Kb + kb) * NT * kKB + ((long long)(kl >> 3) * NT + nl) * 8 + (kl & 7);
            s += fabsf(__half2float(img[at]) + __half2float(img[term + at]));
        }
        s *= 1.0f + 1.0f / 512.0f;
    }
    atomic_max_bits(out, __float_as_uint(s));
}
__global__ void k_tc_scales(const uint32_t* __restrict__ amax, const uint32_t* __restrict__ colsum, int L, int* sexp) {
    float b = __uint_as_float(amax[0]);
    for (int l = L - 1; l >= 0; --l) {
        sexp[l] = scale_exp(b);
        b *= __uint_as_float(colsum[l]);
    }
}
// the forward weight images of one layer (rows n < N, columns k < K) -> its dgrad operand: [term][nt over K, NTd wide][kb over n][n/8][k][n%8]
__global__ void k_tc_transpose_w(const __half* __restrict__ img, int N, int K, int NT, int n_tiles, int Kb, __half* __restrict__ wt, int NTd,
                                 int ntd_tiles, int KbN) {
    const long long total = (long long)N * K, term = (long long)n_tiles * Kb * NT * kKB, term_t = (long long)ntd_tiles * KbN * NTd * kKB;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i / K), k = (int)(i - (long long)n * K);
        const int nt = n / NT, nl = n - nt * NT, kb = k / kKB, kl = k - kb * kKB;
        const long long at = ((long long)nt * Kb + kb) * NT * kKB + ((long long)(kl >> 3) * NT + nl) * 8 + (kl & 7);
        const int td = k / NTd, kd = k - td * NTd, nb = n / kKB, nn = n - nb * kKB;
        const long long att = ((long long)td * KbN + nb) * NTd * kKB + ((long long)(nn >> 3) * NTd + kd) * 8 + (nn & 7);
        wt[att] = img[at];
        wt[term_t + att] = img[term + at];
    }
}
// the head's dZ: dlogits [batch][A] and dvalues [batch] (column A) -> hi / lo images scaled by 2^sexp[0]; zero past the batch and past A (+ 1)
__global__ void k_tc_head_grad(const float* __restrict__ dl, const float* __restrict__ dv, int A, long long batch, int KbZ, const int* __restrict__ sexp,
                               __half* __restrict__ Z, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int row = (int)(i % kM);
    long long r = i / kM;
    const int ch = (int)(r % 8); r /= 8;
    const int kb = (int)(r % KbZ);
    const long long mt = r / KbZ;
    const long long grow = mt * kM + row;
    const int s = __ldg(sexp);
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        float x[2];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int c = kb * kKB + ch * 8 + j + t;
            float v = 0.0f;
            if (grow < batch) {
                if (c < A) v = dl[grow * A + c];
                else if (c == A && dv) v = dv[grow];
            }
            x[t] = ldexpf(v, s);
        }
        const __half h0 = __float2half_rn(x[0]), h1 = __float2half_rn(x[1]);
        const __half l0 = __float2half_rn(x[0] - __half2float(h0)), l1 = __float2half_rn(x[1] - __half2float(h1));
        hi[j >> 1] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
        lo[j >> 1] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
    }
    __half* img = Z + ((size_t)mt * KbZ + kb) * 2 * kImgA + ((size_t)ch * kM + row) * 8;
    *reinterpret_cast<uint4*>(img) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(img + kImgA) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// wgrad:  part[chunk][o][i] = sum over the chunk's rows of dZ[row][o] H[row][i]  (scaled by 2^sexp), tcgen05 with K = rows.
// Both operands are read in place from their images, MN-major: in an image [c/8][row][c%8] a core matrix is 8 rows (K) x 8 contiguous
// columns (MN); K groups of 8 rows are 128 bytes apart (leading byte offset), MN groups of 8 columns 128 x 16 = 2048 bytes (stride byte
// offset).  The two dZ images of a 128-column M tile sit back to back in shared memory, so the MN stride stays 2048 across them.
// Tile = 128 output features (o) x 64 input features (i, one H image); a stage = one 128-row tile: dZ hi / lo of both K blocks (64 KB) + H hi
// (/ lo) (16 / 32 KB); 2 stages.  Products dZ_hi H_hi + dZ_hi H_lo + dZ_lo H_hi (layer 1: H is 0 / 1, exact in hi: two products).
struct WgradArgs {
    const __half* Z; const __half* H; float* part;
    int KbZ, KbH, h_terms, mo_tiles, chunks, m_tiles;
    long long ldp, part_stride;
};
constexpr int kWStages = 2;
constexpr uint32_t kWStageBytes = 6u * kImgA * 2;           // 4 dZ images + 2 H images
constexpr uint32_t kWSmem = kWStages * kWStageBytes + 128;
// MN-major operand descriptor: leading byte offset = K-group stride, stride byte offset = MN-group stride (cute::UMMA canonical INTERLEAVE
// MN-major layout ((8,m),(8,k)) : ((1,SBO),(8,LBO)) in elements)
__host__ __device__ constexpr uint32_t instr_desc_mn(int n) { return instr_desc(n) | (1u << 15) | (1u << 16); }

__global__ void __launch_bounds__(kThreads, 1) k_tc_wgrad(const __grid_constant__ WgradArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* const full = reinterpret_cast<uint64_t*>(smem + kWStages * kWStageBytes);
    uint64_t* const empty = full + kWStages;
    uint64_t* const acc_full = empty + kWStages;
    uint64_t* const acc_empty = acc_full + 2;
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ni_tiles = a.KbH, items = a.chunks * a.mo_tiles * ni_tiles;
    const uint32_t acc_cols = 64;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kWStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(2 * acc_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_launch_dependents();
    pdl_wait();
    // item t -> (chunk, o tile, i tile); the chunk's row tiles [c * kChunkTiles, ..)
    auto decode = [&](int t, int& c, int& mo, int& ni) { ni = t % ni_tiles; t /= ni_tiles; mo = t % a.mo_tiles; c = t / a.mo_tiles; };
    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            const uint32_t bytes = (4u + (uint32_t)a.h_terms) * kImgA * 2;
            for (int t = blockIdx.x; t < items; t += gridDim.x) {
                int c, mo, ni; decode(t, c, mo, ni);
                const int mt1 = min(a.m_tiles, (c + 1) * kChunkTiles);
                for (int mt = c * kChunkTiles; mt < mt1; ++mt) {
                    mbar_wait(empty + stage, phase ^ 1u);
                    mbar_expect_tx(full + stage, bytes);
                    uint8_t* const sp = smem + stage * kWStageBytes;
                    for (int term = 0; term < 2; ++term)             // [term][kb 2 mo, 2 mo + 1]: the M tile's two images back to back
                        for (int j = 0; j < 2; ++j)
                            bulk_g2s(sp + (term * 2 + j) * kImgA * 2, a.Z + (((size_t)mt * a.KbZ + 2 * mo + j) * 2 + term) * kImgA, kImgA * 2, full + stage);
                    for (int term = 0; term < a.h_terms; ++term)
                        bulk_g2s(sp + (4 + term) * kImgA * 2, a.H + (((size_t)mt * a.KbH + ni) * a.h_terms + term) * kImgA, kImgA * 2, full + stage);
                    if (++stage == (uint32_t)kWStages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
        const uint32_t idesc = instr_desc_mn(64), lbo = 128, sbo = 128 * 16;
        for (int t = blockIdx.x; t < items; t += gridDim.x) {
            int c, mo, ni; decode(t, c, mo, ni);
            const int mt1 = min(a.m_tiles, (c + 1) * kChunkTiles);
            mbar_wait(acc_empty + as, aphase ^ 1u);
            tc_fence_after();
            const uint32_t d = tmem_base + as * acc_cols;
            for (int mt = c * kChunkTiles; mt < mt1; ++mt) {
                mbar_wait(full + stage, phase);
                tc_fence_after();
                const uint32_t sp = smem_u32(smem + stage * kWStageBytes);
                const uint32_t z_hi = sp, z_lo = sp + 2 * kImgA * 2, h_hi = sp + 4 * kImgA * 2, h_lo = sp + 5 * kImgA * 2;
#pragma unroll
                for (int k = 0; k < kM / 16; ++k) {                    // K = 16 rows: two 8-row groups, 256 bytes
                    const uint32_t o = 256u * k;
                    umma_f16_w(d, smem_desc(z_hi + o, lbo, sbo), smem_desc(h_hi + o, lbo, sbo), idesc, (mt > c * kChunkTiles || k) ? 1u : 0u);
                    if (a.h_terms == 2) umma_f16_w(d, smem_desc(z_hi + o, lbo, sbo), smem_desc(h_lo + o, lbo, sbo), idesc, 1u);
                    umma_f16_w(d, smem_desc(z_lo + o, lbo, sbo), smem_desc(h_hi + o, lbo, sbo), idesc, 1u);
                }
                umma_commit_w(empty + stage);
                if (++stage == (uint32_t)kWStages) { stage = 0; phase ^= 1u; }
            }
            umma_commit_w(acc_full + as);
            if (++as == 2) { as = 0; aphase ^= 1u; }
        }
    } else {
        const int q = warp & 3, row = q * 32 + lane;
        uint32_t as = 0, aphase = 0;
        for (int t = blockIdx.x; t < items; t += gridDim.x) {
            int c, mo, ni; decode(t, c, mo, ni);
            mbar_wait(acc_full + as, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + as * acc_cols + ((uint32_t)(q * 32) << 16);
            float* dst = a.part + (size_t)c * a.part_stride + (size_t)(mo * kM + row) * a.ldp + (size_t)ni * kKB;
            for (int c0 = 0; c0 < 64; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + (uint32_t)c0, v);
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                    *reinterpret_cast<float4*>(dst + c0 + i) = make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]), __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + as);
            if (++as == 2) { as = 0; aphase ^= 1u; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(2 * acc_cols) : "memory");
}

// db partials: bpart[chunk][o] = sum over the chunk's rows of dZ[row][o] (hi + lo, scaled).  Block = (chunk, K block of dZ), thread = row of a
// tile: 8 tiles in order, then a fixed tree over the 128 rows
__global__ void __launch_bounds__(128) k_tc_bias_partial(const __half* __restrict__ Z, int KbZ, int m_tiles, float* __restrict__ bpart, int ldb) {
    __shared__ float red[128][65];
    const int c = blockIdx.x, kb = blockIdx.y, row = threadIdx.x;
    float s[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) s[j] = 0.0f;
    const int mt1 = min(m_tiles, (c + 1) * kChunkTiles);
    for (int mt = c * kChunkTiles; mt < mt1; ++mt) {
        const __half* img = Z + ((size_t)mt * KbZ + kb) * 2 * kImgA;
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
            const uint4 h = *reinterpret_cast<const uint4*>(img + ((size_t)ch * kM + row) * 8);
            const uint4 l = *reinterpret_cast<const uint4*>(img + kImgA + ((size_t)ch * kM + row) * 8);
            const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&hw[j])), fl = __half22float2(*reinterpret_cast<const __half2*>(&lw[j]));
                s[ch * 8 + 2 * j] += fh.x + fl.x;
                s[ch * 8 + 2 * j + 1] += fh.y + fl.y;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 64; ++j) red[row][j] = s[j];
    __syncthreads();
    for (int w = 64; w >= 1; w >>= 1) {
        if (row < w)
            for (int j = 0; j < 64; ++j) red[row][j] += red[row + w][j];
        __syncthreads();
    }
    if (row < 64) bpart[(size_t)c * ldb + kb * kKB + row] = red[0][row];
}
// partials -> gradients: sum over the chunks in order, times 2^-sexp.  Entry (o, i) of a [rows][ld] partial; o == nrows (the head's column A)
// goes to the value head's gradient
__global__ void k_tc_reduce(const float* __restrict__ part, int chunks, long long stride, long long ld, int nrows, int K, int vrow,
                            const int* __restrict__ sexp, float* __restrict__ out, float* __restrict__ vout) {
    const long long total = (long long)(nrows + vrow) * K;
    const int s = -__ldg(sexp);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int o = (int)(i / K), k = (int)(i - (long long)o * K);
        const float* p = part + (size_t)o * ld + k;
        float acc = 0.0f;
        for (int c = 0; c < chunks; ++c) acc += p[(size_t)c * stride];
        acc = ldexpf(acc, s);
        if (o < nrows) out[i] = acc;
        else vout[k] = acc;
    }
}

}  // namespace tc
}  // namespace qg

using namespace qg;

struct TcLayer {
    int K = 0, N = 0, Kb = 0, NT = 0, n_tiles = 0, Npad = 0, a_terms = 2, relu = 1, stages = qg::tc::kStages, staging = 0;
    __half* W = nullptr; float* bias = nullptr;
};
struct qg_policy_tc {
    bool fused = false;            // three layers that fit k_tc_fused3
    bool force_layers = false;     // qg_policy_tc_set_mode(p, 1): one kernel per layer even where the fused kernel applies (A/B runs, tests)
    __half* W2_fused = nullptr;    // layer 2's weight images with all C_pad rows in one tile
    int device = 0, obs_size = 0, obs_words = 0, num_actions = 0, has_value = 0, num_sms = 148;
    long long max_batch = 0; int m_tiles = 0;
    std::vector<TcLayer> layers;
    std::vector<__half*> acts;     // acts[l] = X images of layer l
    // the last forward (qg_policy_tc_backward refers to it): its generation, batch and whether it ran per layer (acts[] hold its inputs)
    long long generation = 0, fwd_batch = -1; bool fwd_layers = false;
    // qg_policy_tc_enable_training
    bool training = false;
    std::vector<__half*> dz;       // dz[l] = dZ images of layer l [m_tiles][kbz[l]][2][8][128][8]
    std::vector<__half*> wt;       // wt[l] (l >= 1) = the transposed weight images the dgrad reads
    std::vector<int> kbz, ntd;     // dZ K blocks (even) / the dgrad's column tile width of layer l
    float* part = nullptr; float* bpart = nullptr;    // wgrad / db split-K partials
    uint32_t* stats = nullptr;     // [0] amax of the head gradient, [1 + l] colsum of layer l (f32 bits)
    int* sexp = nullptr;           // [l] the power-of-two scale of dZ_l
};

namespace {
#define TC_CUDA_OK(expr)                                                                       \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
            return QG_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline unsigned grid_for(const qg_policy_tc* p, long long total) { return (unsigned)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)p->num_sms * 8)); }

// the dgrad's transposed weight images and the column sums of the scale bound, from the forward weight images (same halves)
int refresh_training_images(qg_policy_tc* p, cudaStream_t st) {
    const int L = (int)p->layers.size();
    TC_CUDA_OK(cudaMemsetAsync(p->stats + 1, 0, sizeof(uint32_t) * L, st));
    for (int l = 0; l < L; ++l) {
        const TcLayer& T = p->layers[l];
        tc::k_tc_colsum<<<(unsigned)((T.K + 255) / 256), 256, 0, st>>>(T.W, T.N, T.K, T.NT, T.n_tiles, T.Kb, p->stats + 1 + l);
        TC_CUDA_OK(cudaGetLastError());
        if (l == 0) continue;
        const int ntd_tiles = p->layers[l - 1].Npad / p->ntd[l];
        tc::k_tc_transpose_w<<<grid_for(p, (long long)T.N * T.K), 256, 0, st>>>(T.W, T.N, T.K, T.NT, T.n_tiles, T.Kb, p->wt[l], p->ntd[l], ntd_tiles, p->kbz[l]);
        TC_CUDA_OK(cudaGetLastError());
    }
    return QG_OK;
}
}  // namespace

extern "C" {

void qg_policy_tc_destroy(qg_policy_tc* p) {
    if (!p) return;
    for (auto& l : p->layers) { if (l.W) cudaFree(l.W); if (l.bias) cudaFree(l.bias); }
    for (auto* a : p->acts) if (a) cudaFree(a);
    if (p->W2_fused) cudaFree(p->W2_fused);
    for (auto* a : p->dz) if (a) cudaFree(a);
    for (auto* a : p->wt) if (a) cudaFree(a);
    if (p->part) cudaFree(p->part);
    if (p->bpart) cudaFree(p->bpart);
    if (p->stats) cudaFree(p->stats);
    if (p->sexp) cudaFree(p->sexp);
    delete p;
}

int qg_policy_tc_create(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features, const float* const* weights_host,
                        const float* const* biases_host, const float* value_weight_host, float value_bias, int64_t max_batch, qg_policy_tc** out) {
    if (!out || !out_features || !weights_host || !biases_host) { set_error("null argument"); return QG_ERR_INVALID; }
    *out = nullptr;
    if (obs_size < 1 || num_layers < 1 || num_layers > 8 || max_batch < 1) { set_error("qg_policy_tc_create: bad sizes"); return QG_ERR_INVALID; }
    int ndev = 0;
    TC_CUDA_OK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { set_error("no such CUDA device (the engine has no CPU fallback)"); return QG_ERR_CUDA; }
    TC_CUDA_OK(cudaSetDevice(device));
    int major = 0;
    TC_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) { set_error("the tensor-core policy needs an sm_100 device (tcgen05)"); return QG_ERR_UNSUPPORTED; }
    qg_policy_tc* p = new (std::nothrow) qg_policy_tc();
    if (!p) { set_error("out of memory"); return QG_ERR_INVALID; }
    p->device = device; p->obs_size = obs_size; p->obs_words = (obs_size + 31) / 32; p->max_batch = max_batch;
    p->m_tiles = (int)((max_batch + tc::kM - 1) / tc::kM);
    p->has_value = value_weight_host ? 1 : 0;
    p->num_actions = out_features[num_layers - 1];
    { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) p->num_sms = v; }
    auto fail = [&](int rc) { qg_policy_tc_destroy(p); return rc; };
    int K = obs_size;
    for (int l = 0; l < num_layers; ++l) {
        TcLayer L;
        const bool last = l == num_layers - 1;
        L.K = K; L.N = out_features[l] + (last ? p->has_value : 0);
        if (out_features[l] < 1 || out_features[l] > 4096) { set_error("qg_policy_tc_create: layer width outside 1..4096"); return fail(QG_ERR_UNSUPPORTED); }
        L.Kb = round_up(K, tc::kKB) / tc::kKB;
        L.a_terms = l == 0 ? 1 : 2; L.relu = last ? 0 : 1;
        if (last) {
            L.Npad = round_up(L.N, 16);
            if (L.Npad > tc::kMaxNT) { set_error("qg_policy_tc_create: more than 127 actions are not supported by the tensor-core head"); return fail(QG_ERR_UNSUPPORTED); }
            L.NT = L.Npad; L.n_tiles = 1;
        } else {
            L.Npad = round_up(L.N, tc::kKB);                      // = the next layer's padded K
            L.NT = (L.Npad % 128 == 0) ? 128 : 64; L.n_tiles = L.Npad / L.NT;
        }
        // weight tile images [term][n_tile][kb][k/8][n][k%8], halves; zero padding rows / columns
        const size_t img = (size_t)L.NT * tc::kKB, count = (size_t)2 * L.n_tiles * L.Kb * img;
        std::vector<__half> wimg(count, __float2half(0.0f));
        std::vector<float> bias((size_t)L.Npad, 0.0f);
        const float* W = weights_host[l];
        for (int n = 0; n < L.N; ++n) {
            const bool vrow = last && p->has_value && n == out_features[l];
            bias[n] = vrow ? value_bias : biases_host[l][n];
            const float* wr = vrow ? value_weight_host : W + (size_t)n * K;
            const int nt = n / L.NT, nl = n % L.NT;
            for (int k = 0; k < K; ++k) {
                const float w = wr[k];
                const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
                const int kb = k / tc::kKB, kl = k % tc::kKB;
                const size_t at = (((size_t)nt * L.Kb + kb) * img) + ((size_t)(kl >> 3) * L.NT + nl) * 8 + (kl & 7);
                wimg[at] = hi;
                wimg[(size_t)L.n_tiles * L.Kb * img + at] = lo;
            }
        }
        cudaError_t ce = cudaMalloc(&L.W, count * sizeof(__half));
        if (ce == cudaSuccess) ce = cudaMemcpy(L.W, wimg.data(), count * sizeof(__half), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMalloc(&L.bias, bias.size() * 4);
        if (ce == cudaSuccess) ce = cudaMemcpy(L.bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice);
        p->layers.push_back(L);
        if (ce != cudaSuccess) { set_error(std::string("qg_policy_tc_create: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
        // this layer's input images
        __half* X = nullptr;
        const size_t xbytes = (size_t)p->m_tiles * L.Kb * L.a_terms * tc::kImgA * sizeof(__half);
        ce = cudaMalloc(&X, xbytes);
        if (ce == cudaSuccess) ce = cudaMemset(X, 0, xbytes);
        p->acts.push_back(X);
        if (ce != cudaSuccess) { set_error(std::string("qg_policy_tc_create: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
        K = out_features[l];
    }
    // (layer l writes round_up(N_l, 64) columns = all K blocks of layer l+1: padded columns come out as relu(0 + 0) = 0)
    size_t max_smem = 0;
    for (size_t l = 0; l < p->layers.size(); ++l) {
        TcLayer& L = p->layers[l];
        L.staging = (l + 1 == p->layers.size()) ? tc::kM * p->num_actions : 0;
        L.stages = tc::kStages;
        while (L.stages > 1 && tc::plan_smem(L.a_terms, L.NT, L.stages, L.staging).total > 220 * 1024) --L.stages;
        max_smem = std::max<size_t>(max_smem, tc::plan_smem(L.a_terms, L.NT, L.stages, L.staging).total);
    }
    cudaError_t ce = cudaFuncSetAttribute(tc::k_tc_layer<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem);
    if (ce != cudaSuccess) { set_error(std::string("qg_policy_tc_create: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
    // the one-kernel path: embeddings (a multiple of 128 wide after padding) -> one common layer (<= 256) -> head
    if (num_layers == 3 && p->layers[0].Npad % 128 == 0 && p->layers[0].Npad <= 512 && p->layers[0].NT == 128 && p->layers[1].Npad <= 256) {
        const TcLayer& L1 = p->layers[1];
        const int C_pad = L1.Npad, Kb2 = L1.Kb, K = L1.K;
        const size_t img = (size_t)C_pad * tc::kKB, count = (size_t)2 * Kb2 * img;
        std::vector<__half> wimg(count, __float2half(0.0f));
        const float* W = weights_host[1];
        for (int n = 0; n < out_features[1]; ++n)
            for (int k = 0; k < K; ++k) {
                const float w = W[(size_t)n * K + k];
                const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
                const int kb = k / tc::kKB, kl = k % tc::kKB;
                const size_t at = (size_t)kb * img + ((size_t)(kl >> 3) * C_pad + n) * 8 + (kl & 7);
                wimg[at] = hi; wimg[(size_t)Kb2 * img + at] = lo;
            }
        ce = cudaMalloc(&p->W2_fused, count * sizeof(__half));
        if (ce == cudaSuccess) ce = cudaMemcpy(p->W2_fused, wimg.data(), count * sizeof(__half), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaFuncSetAttribute(tc::k_tc_fused3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kFusedSmem);
        if (ce != cudaSuccess) { set_error(std::string("qg_policy_tc_create: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
        p->fused = true;
    }
    *out = p;
    return QG_OK;
}

int qg_policy_tc_load_weights_dev(qg_policy_tc* p, int32_t obs_size, int32_t num_layers, const int32_t* out_features, const float* const* weights_dev,
                                  const float* const* biases_dev, const float* value_weight_dev, const float* value_bias_dev, qg_stream stream) {
    if (!p || !out_features || !weights_dev || !biases_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (obs_size != p->obs_size || num_layers != (int)p->layers.size()) { set_error("qg_policy_tc_load_weights_dev: shapes differ from creation"); return QG_ERR_INVALID; }
    if ((value_weight_dev != nullptr) != (p->has_value != 0) || (value_weight_dev && !value_bias_dev)) {
        set_error("qg_policy_tc_load_weights_dev: the value head must be given exactly when the handle was created with one");
        return QG_ERR_INVALID;
    }
    for (int l = 0; l < num_layers; ++l) {
        const TcLayer& L = p->layers[l];
        const int rows = L.N - ((l == num_layers - 1) ? p->has_value : 0);
        if (out_features[l] != rows || !weights_dev[l] || !biases_dev[l]) { set_error("qg_policy_tc_load_weights_dev: shapes differ from creation"); return QG_ERR_INVALID; }
    }
    TC_CUDA_OK(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    auto grid_for = [&](long long total) { return (unsigned)std::min<long long>((total + 255) / 256, (long long)p->num_sms * 8); };
    for (int l = 0; l < num_layers; ++l) {
        const TcLayer& L = p->layers[l];
        const bool last = l == num_layers - 1;
        const float* vw = (last && p->has_value) ? value_weight_dev : nullptr;
        tc::k_tc_load_layer<<<grid_for((long long)L.N * L.K), 256, 0, st>>>(weights_dev[l], biases_dev[l], vw, value_bias_dev, out_features[l], L.K, L.NT,
                                                                         L.n_tiles, L.Kb, L.W, L.bias);
        TC_CUDA_OK(cudaGetLastError());
    }
    if (p->W2_fused) {          // the fused kernel's copy of layer 2: all C_pad rows in one tile
        const TcLayer& L1 = p->layers[1];
        tc::k_tc_load_layer<<<grid_for((long long)out_features[1] * L1.K), 256, 0, st>>>(weights_dev[1], nullptr, nullptr, nullptr, out_features[1], L1.K,
                                                                                       L1.Npad, 1, L1.Kb, p->W2_fused, nullptr);
        TC_CUDA_OK(cudaGetLastError());
    }
    return p->training ? refresh_training_images(p, st) : QG_OK;
}

int32_t qg_policy_tc_num_actions(const qg_policy_tc* p) { return p ? p->num_actions : 0; }
int32_t qg_policy_tc_set_mode(qg_policy_tc* p, int32_t per_layer) {
    if (!p) return 0;
    p->force_layers = per_layer != 0;
    return (p->fused && !p->force_layers) ? 1 : 0;
}

int qg_policy_tc_forward_bits(qg_policy_tc* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev, float* logits_dev, float* values_dev,
                              qg_stream stream) {
    if (!p || !obs_bits_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (batch < 0 || batch > p->max_batch) { set_error("qg_policy_tc_forward_bits: batch larger than the handle was created for"); return QG_ERR_INVALID; }
    if (values_dev && !p->has_value) { set_error("qg_policy_tc_forward_bits: the policy has no value head"); return QG_ERR_INVALID; }
    ++p->generation; p->fwd_batch = batch; p->fwd_layers = !(p->fused && !p->force_layers);
    if (batch == 0) return QG_OK;
    TC_CUDA_OK(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int m_tiles = (int)((batch + tc::kM - 1) / tc::kM);
    if (!(p->fused && !p->force_layers)) {          // (the fused kernel expands the bits itself)
        const TcLayer& L0 = p->layers[0];
        const long long total = (long long)m_tiles * L0.Kb * 8 * tc::kM;
        tc::k_tc_expand_bits<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(obs_bits_dev, p->obs_words, p->obs_size, batch, L0.Kb, p->acts[0], total);
        TC_CUDA_OK(cudaGetLastError());
    }
    if (p->fused && !p->force_layers) {
        const TcLayer &L0 = p->layers[0], &L1 = p->layers[1], &L2 = p->layers[2];
        tc::FusedArgs a{};
        a.bits = obs_bits_dev; a.obs_words = p->obs_words; a.obs_size = p->obs_size;
        a.X0 = p->acts[0]; a.W1 = L0.W; a.W2 = p->W2_fused; a.W3 = L2.W; a.b1 = L0.bias; a.b2 = L1.bias; a.b3 = L2.bias;
        a.logits = logits_dev; a.probs = probs_dev; a.values = values_dev;
        a.Kb0 = L0.Kb; a.NC = L0.Npad / 128; a.C_pad = L1.Npad; a.Kb3 = L2.Kb; a.H = L2.Npad; a.m_tiles = m_tiles;
        a.num_actions = p->num_actions; a.has_value = p->has_value; a.batch = batch;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3((unsigned)std::min(m_tiles, p->num_sms)); lc.blockDim = dim3(tc::kFusedThreads);
        lc.dynamicSmemBytes = tc::kFusedSmem; lc.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = at; lc.numAttrs = 1;
        TC_CUDA_OK(cudaLaunchKernelEx(&lc, tc::k_tc_fused3, a));
        return QG_OK;
    }
    for (size_t l = 0; l < p->layers.size(); ++l) {
        const TcLayer& L = p->layers[l];
        const bool last = l + 1 == p->layers.size();
        tc::LayerArgs a{};
        a.X = p->acts[l]; a.W = L.W; a.bias = L.bias; a.Y = last ? nullptr : p->acts[l + 1];
        a.logits = last ? logits_dev : nullptr; a.probs = last ? probs_dev : nullptr; a.values = last ? values_dev : nullptr;
        a.a_terms = L.a_terms; a.Kb = L.Kb; a.NT = L.NT; a.n_tiles = L.n_tiles; a.m_tiles = m_tiles;
        a.out_Kb = last ? 0 : p->layers[l + 1].Kb; a.relu = L.relu; a.num_actions = p->num_actions; a.has_value = p->has_value; a.batch = batch;
        a.stages = L.stages;
        const int tiles = m_tiles * L.n_tiles;
        // programmatic dependent launch: the kernel's prologue (barrier init, tensor-memory allocation) overlaps the previous kernel's tail;
        // it waits (griddepcontrol.wait) before it touches global memory
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3((unsigned)std::min(tiles, p->num_sms)); lc.blockDim = dim3(tc::kThreads);
        lc.dynamicSmemBytes = tc::plan_smem(L.a_terms, L.NT, L.stages, L.staging).total; lc.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = at; lc.numAttrs = 1;
        TC_CUDA_OK(cudaLaunchKernelEx(&lc, tc::k_tc_layer<0>, a));
    }
    return QG_OK;
}

int64_t qg_policy_tc_generation(const qg_policy_tc* p) { return p ? p->generation : 0; }

int qg_policy_tc_enable_training(qg_policy_tc* p) {
    if (!p) { set_error("null argument"); return QG_ERR_INVALID; }
    if (p->training) return QG_OK;
    TC_CUDA_OK(cudaSetDevice(p->device));
    const int L = (int)p->layers.size();
    const int chunks = (p->m_tiles + tc::kChunkTiles - 1) / tc::kChunkTiles;
    p->dz.assign(L, nullptr); p->wt.assign(L, nullptr); p->kbz.assign(L, 0); p->ntd.assign(L, 0);
    size_t part_floats = 0, bpart_floats = 0;
    for (int l = 0; l < L; ++l) {
        const TcLayer& T = p->layers[l];
        p->kbz[l] = round_up((T.Npad + tc::kKB - 1) / tc::kKB, 2);
        const size_t zbytes = (size_t)p->m_tiles * p->kbz[l] * 2 * tc::kImgA * sizeof(__half);
        TC_CUDA_OK(cudaMalloc(&p->dz[l], zbytes));
        TC_CUDA_OK(cudaMemset(p->dz[l], 0, zbytes));      // (K blocks past the layer's width are never written: they stay zero)
        part_floats = std::max(part_floats, (size_t)chunks * p->kbz[l] * tc::kKB * T.Kb * tc::kKB);
        bpart_floats = std::max(bpart_floats, (size_t)chunks * p->kbz[l] * tc::kKB);
        if (l == 0) continue;
        const int kpad = p->layers[l - 1].Npad;             // the dgrad's output columns: layer l's input, padded to 64
        p->ntd[l] = kpad % 128 == 0 ? 128 : 64;
        const size_t wbytes = (size_t)2 * (kpad / p->ntd[l]) * p->kbz[l] * p->ntd[l] * tc::kKB * sizeof(__half);
        TC_CUDA_OK(cudaMalloc(&p->wt[l], wbytes));
        TC_CUDA_OK(cudaMemset(p->wt[l], 0, wbytes));
    }
    TC_CUDA_OK(cudaFuncSetAttribute(tc::k_tc_layer<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::plan_smem(2, 128, tc::kStages, 0).total));
    TC_CUDA_OK(cudaMalloc(&p->part, part_floats * sizeof(float)));
    TC_CUDA_OK(cudaMalloc(&p->bpart, bpart_floats * sizeof(float)));
    TC_CUDA_OK(cudaMalloc(&p->stats, sizeof(uint32_t) * (1 + L)));
    TC_CUDA_OK(cudaMalloc(&p->sexp, sizeof(int) * L));
    TC_CUDA_OK(cudaFuncSetAttribute(tc::k_tc_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kWSmem));
    p->training = true;
    const int rc = refresh_training_images(p, nullptr);
    if (rc != QG_OK) return rc;
    TC_CUDA_OK(cudaDeviceSynchronize());
    return QG_OK;
}

int qg_policy_tc_backward(qg_policy_tc* p, int64_t generation, int64_t batch, const float* dlogits_dev, const float* dvalues_dev, float* const* grad_w_dev,
                          float* const* grad_b_dev, float* grad_vw_dev, float* grad_vb_dev, qg_stream stream) {
    if (!p || !dlogits_dev || !grad_w_dev || !grad_b_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (!p->training) { set_error("qg_policy_tc_backward: qg_policy_tc_enable_training was not called"); return QG_ERR_INVALID; }
    if (generation != p->generation || batch != p->fwd_batch || !p->fwd_layers) {
        set_error("qg_policy_tc_backward: not the handle's latest forward (a newer forward ran, or the latest ran the fused kernel)");
        return QG_ERR_INVALID;
    }
    if (p->has_value && (!grad_vw_dev || !grad_vb_dev)) { set_error("qg_policy_tc_backward: the value head's gradient buffers are missing"); return QG_ERR_INVALID; }
    const int L = (int)p->layers.size();
    for (int l = 0; l < L; ++l) if (!grad_w_dev[l] || !grad_b_dev[l]) { set_error("null argument"); return QG_ERR_INVALID; }
    if (batch == 0) return QG_OK;
    TC_CUDA_OK(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int m_tiles = (int)((batch + tc::kM - 1) / tc::kM);
    const int chunks = (m_tiles + tc::kChunkTiles - 1) / tc::kChunkTiles;
    const int A = p->num_actions;
    // scales: amax of the head's gradient, then the bound chain (k_tc_scales)
    TC_CUDA_OK(cudaMemsetAsync(p->stats, 0, sizeof(uint32_t), st));
    const long long n_dl = batch * A, n_dv = dvalues_dev ? batch : 0;
    tc::k_tc_amax<<<grid_for(p, n_dl + n_dv), 256, 0, st>>>(dlogits_dev, n_dl, dvalues_dev, n_dv, p->stats);
    TC_CUDA_OK(cudaGetLastError());
    tc::k_tc_scales<<<1, 1, 0, st>>>(p->stats, p->stats + 1, L, p->sexp);
    TC_CUDA_OK(cudaGetLastError());
    {
        const long long total = (long long)m_tiles * p->kbz[L - 1] * 8 * tc::kM;
        tc::k_tc_head_grad<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(dlogits_dev, p->has_value ? dvalues_dev : nullptr, A, batch, p->kbz[L - 1],
                                                                             p->sexp + (L - 1), p->dz[L - 1], total);
        TC_CUDA_OK(cudaGetLastError());
    }
    // dgrad, layers L .. 2: dZ_(l-1) = mask_l (dZ_l W_l) 2^(s_(l-1) - s_l)
    for (int l = L - 1; l >= 1; --l) {
        const int kpad = p->layers[l - 1].Npad, NT = p->ntd[l];
        tc::LayerArgs a{};
        a.X = p->dz[l]; a.W = p->wt[l]; a.bias = nullptr; a.Y = p->dz[l - 1];
        a.a_terms = 2; a.Kb = p->kbz[l]; a.NT = NT; a.n_tiles = kpad / NT; a.m_tiles = m_tiles; a.out_Kb = p->kbz[l - 1];
        a.relu = 0; a.num_actions = A; a.has_value = 0; a.batch = batch; a.stages = tc::kStages;
        a.mask = p->acts[l]; a.sexp = p->sexp; a.s_in = l; a.s_out = l - 1; a.mask_Kb = p->layers[l].Kb;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3((unsigned)std::min(m_tiles * a.n_tiles, p->num_sms)); lc.blockDim = dim3(tc::kThreads);
        lc.dynamicSmemBytes = tc::plan_smem(2, NT, tc::kStages, 0).total; lc.stream = st;
        TC_CUDA_OK(cudaLaunchKernelEx(&lc, tc::k_tc_layer<1>, a));
    }
    // wgrad and db of every layer: split-K partials per 1024-row chunk, reduced in chunk order
    for (int l = 0; l < L; ++l) {
        const TcLayer& T = p->layers[l];
        const bool last = l == L - 1;
        const int nrows = T.N - (last ? p->has_value : 0), vrow = last ? p->has_value : 0;
        tc::WgradArgs w{};
        w.Z = p->dz[l]; w.H = p->acts[l]; w.part = p->part;
        w.KbZ = p->kbz[l]; w.KbH = T.Kb; w.h_terms = T.a_terms; w.mo_tiles = p->kbz[l] / 2; w.chunks = chunks; w.m_tiles = m_tiles;
        w.ldp = (long long)T.Kb * tc::kKB; w.part_stride = (long long)p->kbz[l] * tc::kKB * w.ldp;
        const int items = chunks * w.mo_tiles * w.KbH;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3((unsigned)std::min(items, p->num_sms)); lc.blockDim = dim3(tc::kThreads);
        lc.dynamicSmemBytes = tc::kWSmem; lc.stream = st;
        TC_CUDA_OK(cudaLaunchKernelEx(&lc, tc::k_tc_wgrad, w));
        tc::k_tc_reduce<<<grid_for(p, (long long)T.N * T.K), 256, 0, st>>>(p->part, chunks, w.part_stride, w.ldp, nrows, T.K, vrow, p->sexp + l,
                                                                           grad_w_dev[l], grad_vw_dev);
        TC_CUDA_OK(cudaGetLastError());
        const int ldb = p->kbz[l] * tc::kKB;
        tc::k_tc_bias_partial<<<dim3((unsigned)chunks, (unsigned)p->kbz[l]), 128, 0, st>>>(p->dz[l], p->kbz[l], m_tiles, p->bpart, ldb);
        TC_CUDA_OK(cudaGetLastError());
        tc::k_tc_reduce<<<grid_for(p, T.N), 256, 0, st>>>(p->bpart, chunks, ldb, 1, nrows, 1, vrow, p->sexp + l, grad_b_dev[l], grad_vb_dev);
        TC_CUDA_OK(cudaGetLastError());
    }
    return QG_OK;
}

}  // extern "C"

#ifdef QG_TC_PROBE
// tools build: [160 CTAs][8] cycle counters of the last fused launch (see g_tc_wait / g_tc_epi)
extern "C" __attribute__((visibility("default"))) int qg_policy_tc_debug_read(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, qg::tc::g_tc_wait, sizeof(long long) * 160 * 8) == cudaSuccess ? 0 : -1;
}
extern "C" __attribute__((visibility("default"))) int qg_policy_tc_debug_read_epilogue(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, qg::tc::g_tc_epi, sizeof(long long) * 160 * 8) == cudaSuccess ? 0 : -1;
}
#endif
