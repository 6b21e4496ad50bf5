// qg_search_fused.cuh — the whole synth-time rollout search of a CTA's rollouts in ONE kernel (DESIGN.md §3 "Search").
//
// Rollouts are independent, so a CTA that owns 8 of them never has to talk to another CTA: per decision it evaluates the policy for
// its 8 packed observations (policy_forward_rows: 8 compute warps + the weight-streaming producer warp), then warp 0 plays the
// sampled / arg-max actions on its 8 environments with the same step_tile<KIND, MODE_SEARCH> the two-kernel path launches,
// which writes the next packed observations; it loops until its rollouts are all final or the decision budget is spent.  No
// launch gaps, no host round trips: a search is one launch.  The first layer's exact integer accumulators stay in global memory
// (L2) between decisions and are only updated with the observation entries the step changed (layer0_fixed); since that sum is order
// independent, the decisions are bit for bit those of the two-kernel path, which sums every set entry afresh.
#pragma once
#include <cstdio>
#include "qg_kernels.cuh"
#include "qg_policy_kernels.cuh"

namespace qg {

static_assert(kStride == 33, "layer0_fixed (qg_policy_kernels.cuh) reads the step's bit stream with a word stride of 33");

template <int KIND>
__global__ void __launch_bounds__(kPolThreads) k_search_fused(const __grid_constant__ DevCfg c, const __grid_constant__ StepArgs a, const __grid_constant__ PolicyDev p,
                                                               int max_decisions, int32_t* __restrict__ decisions_out, long long* __restrict__ acc0_all,
                                                               const uint32_t* __restrict__ first_bits) {
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
        policy_forward_rows(p, ps, it == 0 ? first_bits : nullptr, row0, c.B, s_probs, nullptr, G, it, 0, acc0, obs_stream, cnt);
        __syncthreads();
        { QG_SP_T0();
        if (warp == 0) {
            const uint32_t en = step_tile<KIND, MODE_SEARCH, 0, 32, 0, false>(c, a, wbase, nullptr, lane, row0, cnt, it > 0, s_probs, true, s_ret);
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

template <int KIND>
cudaError_t launch_search_fused(const DevCfg& c, const StepArgs& a, const PolicyDev& p, int max_decisions, int32_t* decisions_out, size_t step_smem_bytes, long long* acc0,
                                const uint32_t* first_bits, cudaStream_t st) {
    const size_t smem = policy_smem_bytes(p) + step_smem_bytes + (size_t)kPolRows * p.num_actions * 4;
    cudaError_t e = cudaFuncSetAttribute(k_search_fused<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((c.B + kPolRows - 1) / kPolRows);
    k_search_fused<KIND><<<grid, kPolThreads, smem, st>>>(c, a, p, max_decisions, decisions_out, acc0, first_bits);
    return cudaGetLastError();
}

}  // namespace qg
