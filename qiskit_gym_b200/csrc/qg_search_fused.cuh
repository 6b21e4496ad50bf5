// qg_search_fused.cuh — the whole synth-time rollout search of a CTA's rollouts in ONE kernel (DESIGN.md §3 "Search").
//
// Rollouts are independent, so a CTA that owns 8 of them never has to talk to another CTA: per decision it evaluates the policy for
// its 8 packed observations (policy_forward_rows: 8 compute warps + the weight-streaming producer warp), then warp 0 plays the
// sampled / arg-max actions on its 8 environments with the same step_tile<KIND, MODE_SEARCH> the two-kernel path launches,
// which writes the next packed observations; it loops until its rollouts are all final or the decision budget is spent.  No
// launch gaps, no host round trips: a search is one launch.  The first layer's exact integer accumulators stay in global memory
// (L2) between decisions and are only updated with the observation entries the step changed (layer0_fixed); since that sum is order
// independent, the decisions are bit for bit those of the two-kernel path, which sums every set entry afresh.
//
// TWIST (qg_search_run_twisted): the twisted search.  Protocol (DESIGN.md §3 "Twisted search"): at every decision rollout i (global id
// g = first_id + i) runs the policy in frame k = mulhi(philox(seed; g, tick, STREAM_TWIST), K) of the env's K twists, tick = its step
// counter HD_TICK at decision time (the counter that also keys the decision's sample draw), so k depends on the seed, g and the decision
// index only.  The policy sees the observation in frame k (entry i moves to obs_perms[k][i], twist_word); env action a weighs
// probs[act_perm[k][a]] and the arg-max / inverse-CDF sum run over a in env order (step_tile's TWIST path).  Solutions, returns and keys
// are those of the env.  The first decision reads the twisted observation qg_search_observe_twisted wrote (and its k in tw.twist); every
// later one twists the CTA's 8 rows of the step's shared-memory bit stream into the policy's row buffer (ps.rowbits) and writes k to
// tw.twist, where the step reads it.  layer0_fixed keeps its accumulators incremental: it diffs whatever rows it is given against the
// previous pass, and the sum is exact, so the frame changing between decisions only changes how many entries it updates.
#pragma once
#include <cstdio>
#include "qg_kernels.cuh"
#include "qg_launch.hpp"
#include "qg_policy_kernels.cuh"

namespace qg {

static_assert(kStride == 33, "layer0_fixed (qg_policy_kernels.cuh) reads the step's bit stream with a word stride of 33");

template <int KIND, bool TWIST = false>
__global__ void __launch_bounds__(kPolThreads) k_search_fused(const __grid_constant__ DevCfg c, const __grid_constant__ StepArgs a, const __grid_constant__ PolicyDev p,
                                                               int max_decisions, int32_t* __restrict__ decisions_out, long long* __restrict__ acc0_all,
                                                               const uint32_t* __restrict__ first_bits, const __grid_constant__ SearchTwist tw) {
    extern __shared__ __align__(128) float smf[];
    __shared__ uint32_t s_active;
    __shared__ float s_ret[kPolRows];              // running returns of the CTA's rollouts (Env::reward summed in step order)
    const PolicySmem ps = policy_smem_carve(p, smf);
    uint32_t* const wbase = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(smf) + policy_smem_bytes(p));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * kPolRows;
    const int cnt = (int)min((int64_t)kPolRows, c.B - row0);
    float* const s_probs = reinterpret_cast<float*>(wbase + a.sm_warp_words);      // [kPolRows][A] action weights of the CTA's rollouts
    const bool obs_from_O = (KIND == QG_ENV_PAULI_NETWORK) || (KIND == QG_ENV_PERMUTATION && c.OW > 0);
    const uint32_t* const obs_stream = wbase + (obs_from_O ? a.sm_obs : c.off_state * kStride);   // the step's [word][env] observation bit stream
    long long* const acc0 = acc0_all + (size_t)blockIdx.x * kPolRows * p.width[0];     // this CTA's first-layer accumulators
    policy_init_barriers(ps, tid);
    if (tid < kPolRows) s_ret[tid] = tid < cnt ? c.ret[row0 + tid] : 0.0f;
    __syncthreads();
    int G = 0, it = 0;
#ifdef QG_SEARCH_PROBE
    const long long sp_total0 = clock64();
#endif
    for (; it < max_decisions; ++it) {
        // decision `it`: the first one reads the packed observations qg_observe_bits left in global memory, the later ones read the
        // step's own bit stream in shared memory; the action weights stay in shared memory; the env records stay in the step's region
        if constexpr (TWIST) {
            if (it > 0) {
                // rows of this decision's frame into ps.rowbits: thread = (row, word); k from the row's resident tick
                const int OW = p.obs_words;
                for (int i = tid; i < kPolRows * OW; i += kPolThreads) {
                    const int r = i / OW, w = i - r * OW;
                    uint32_t v = 0;
                    if (r < cnt) {
                        const uint32_t k = twist_draw(seed_of(c), c.first_id + row0 + r, wbase[HD_TICK * kStride + r], tw.K);
                        if (w == 0) tw.twist[row0 + r] = (int32_t)k;
                        v = twist_word([&](int s) { return (obs_stream[(s >> 5) * kStride + r] >> (s & 31)) & 1u; }, w, c.obs_size, c.n, tw.d,
                                       tw.qpinv + (size_t)k * c.n);
                    }
                    ps.rowbits[i] = v;
                }
                __syncthreads();
            }
            policy_forward_rows(p, ps, it == 0 ? first_bits : nullptr, row0, c.B, s_probs, nullptr, G, it, 0, acc0, nullptr, 0);
        } else {
            policy_forward_rows(p, ps, it == 0 ? first_bits : nullptr, row0, c.B, s_probs, nullptr, G, it, 0, acc0, obs_stream, cnt);
        }
        __syncthreads();
        { QG_SP_T0();
        if (warp == 0) {
            const uint32_t en = step_tile<KIND, MODE_SEARCH, 0, 32, 0, TWIST>(c, a, wbase, nullptr, lane, row0, cnt, it > 0, s_probs, true, s_ret);
            if (lane == 0) s_active = en;
        }
        __syncthreads();                           // next observations in the step's stream, s_active set
        QG_SP_ADD(10); }
#ifdef QG_SEARCH_PROBE
        if (threadIdx.x == 0 && blockIdx.x == 0) g_search_prof[11] += 1;
#endif
        if (s_active == 0) break;                  // every rollout of this CTA is final
    }
#ifdef QG_SEARCH_PROBE
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        g_search_prof[12] += clock64() - sp_total0;
        printf("SEARCHPROF obs %lld l0 %lld l1 %lld l2 %lld l3 %lld softmax %lld step %lld decisions %lld total %lld\n", g_search_prof[0], g_search_prof[1], g_search_prof[2],
               g_search_prof[3], g_search_prof[4], g_search_prof[9], g_search_prof[10], g_search_prof[11], g_search_prof[12]);
        for (int i = 0; i < 16; ++i) g_search_prof[i] = 0;
    }
#endif
    if (warp == 0) {                               // what stayed in shared memory during the search goes back: records, returns
        tile_writeback(c, wbase, lane, row0, cnt);
        if (lane < cnt) c.ret[row0 + lane] = s_ret[lane];
    }
    if (tid == 0 && decisions_out) decisions_out[blockIdx.x] = min(it + 1, max_decisions);
}

// Dynamic shared memory one k_search_fused CTA asks for: the policy's plan, one warp region of the step kernel and the CTA's action
// weights (s_probs, [kPolRows][A] floats).  launch_search_fused requests exactly this; search_fused_smem checks it against the device.
inline size_t search_fused_dynamic_smem(const PolicyDev& p, size_t step_smem_bytes) {
    return policy_smem_bytes(p) + step_smem_bytes + (size_t)kPolRows * p.num_actions * 4;
}

template <int KIND, bool TWIST>
cudaError_t search_fused_smem(const PolicyDev& p, size_t step_smem_bytes, int device, size_t* dynamic_bytes, size_t* static_bytes, size_t* limit) {
    cudaFuncAttributes fa{};
    // (PauliNetwork has no twisted search: its symmetry is applied inside the env; its TWIST instantiation is never built)
    cudaError_t e = cudaFuncGetAttributes(&fa, k_search_fused<KIND, TWIST && KIND != QG_ENV_PAULI_NETWORK>);
    int optin = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    *dynamic_bytes = search_fused_dynamic_smem(p, step_smem_bytes);
    *static_bytes = fa.sharedSizeBytes;                 // the kernel's s_active / s_ret
    *limit = (size_t)optin;
    return e;
}

// tw: null for the untwisted search (k_search_fused<KIND, false>), the tables of the twisted one otherwise.
template <int KIND>
cudaError_t launch_search_fused(const DevCfg& c, const StepArgs& a, const PolicyDev& p, int max_decisions, int32_t* decisions_out, size_t step_smem_bytes, long long* acc0,
                                const uint32_t* first_bits, const SearchTwist* tw, cudaStream_t st) {
    const size_t smem = search_fused_dynamic_smem(p, step_smem_bytes);
    const unsigned grid = (unsigned)((c.B + kPolRows - 1) / kPolRows);
    if (tw) {
        if constexpr (KIND == QG_ENV_PAULI_NETWORK) return cudaErrorNotSupported;
        else {
            cudaError_t e = cudaFuncSetAttribute(k_search_fused<KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            k_search_fused<KIND, true><<<grid, kPolThreads, smem, st>>>(c, a, p, max_decisions, decisions_out, acc0, first_bits, *tw);
            return cudaGetLastError();
        }
    }
    cudaError_t e = cudaFuncSetAttribute(k_search_fused<KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_search_fused<KIND, false><<<grid, kPolThreads, smem, st>>>(c, a, p, max_decisions, decisions_out, acc0, first_bits, SearchTwist{});
    return cudaGetLastError();
}

}  // namespace qg
