// qg_step_kind.cuh — definitions behind qg_launch.hpp; included by the per-kind translation units only.
#pragma once
#include <cstdlib>

#include "qg_launch.hpp"
#include "qg_search_fused.cuh"

namespace qg {

template <int KIND, int MODE, int INV, int EPW>
cudaError_t launch_epw(const DevCfg& c, const StepArgs& a, const LaunchGeom& g, cudaStream_t st) {
    // programmatic dependent launch: the grid may start while its predecessor in the stream drains; the kernel
    // waits (griddepcontrol.wait) before it touches the records
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(g.grid); lc.blockDim = dim3(kWarpsPerCta * 32); lc.dynamicSmemBytes = g.smem_bytes; lc.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (g.pdl) { at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
    if (g.l2_bytes > 0) {
        at[na].id = cudaLaunchAttributeAccessPolicyWindow;
        at[na].val.accessPolicyWindow.base_ptr = const_cast<void*>(g.l2_base);
        at[na].val.accessPolicyWindow.num_bytes = g.l2_bytes;
        at[na].val.accessPolicyWindow.hitRatio = 1.0f;
        at[na].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        at[na].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        ++na;
    }
    lc.attrs = at; lc.numAttrs = na;
    if constexpr (MODE == MODE_STEP && EPW == 32) { if (a.pair) return cudaLaunchKernelEx(&lc, k_step<KIND, MODE, INV, EPW, 1>, c, a); }
    return cudaLaunchKernelEx(&lc, k_step<KIND, MODE, INV, EPW, 0>, c, a);
}

template <int KIND, int MODE, int INV>
cudaError_t launch_one(const DevCfg& c, const StepArgs& a, const LaunchGeom& g, cudaStream_t st) {
    // 16-env tiles exist for the stepping modes only (MODE_OBSERVE launches are rare reads)
    if constexpr (MODE != MODE_OBSERVE) { if (g.epw == 16) return launch_epw<KIND, MODE, INV, 16>(c, a, g, st); }
    return launch_epw<KIND, MODE, INV, 32>(c, a, g, st);
}

constexpr bool kind_has_matrix_inverse(int kind) { return kind == QG_ENV_LINEAR_FUNCTION || kind == QG_ENV_CLIFFORD; }

template <int KIND, int MODE>
cudaError_t launch_mode(int inv, const DevCfg& c, const StepArgs& a, const LaunchGeom& g, cudaStream_t st) {
    if constexpr (kind_has_matrix_inverse(KIND) && MODE != MODE_OBSERVE) {
        switch (inv) {
            case 8: return launch_one<KIND, MODE, 8>(c, a, g, st);
            case 16: return launch_one<KIND, MODE, 16>(c, a, g, st);
            case 32: return launch_one<KIND, MODE, 32>(c, a, g, st);
            default: break;
        }
    }
    return launch_one<KIND, MODE, 0>(c, a, g, st);
}

template <int KIND>
cudaError_t launch_step_kind(int mode, int inv, const DevCfg& c, const StepArgs& a, const LaunchGeom& g, cudaStream_t st) {
    switch (mode) {
        case MODE_STEP: return launch_mode<KIND, MODE_STEP>(inv, c, a, g, st);
        case MODE_SEARCH: return launch_mode<KIND, MODE_SEARCH>(inv, c, a, g, st);
        default: return launch_mode<KIND, MODE_OBSERVE>(0, c, a, g, st);
    }
}

template <int KIND, int MODE, int INV>
cudaError_t prepare_one(size_t smem_bytes) {
    // same shared-memory carve-out as the policy kernel (qg_policy.cu): alternating launches of the two in a search do not make
    // the SMs reconfigure their L1 / shared-memory split in between
    int carve = (int)cudaSharedmemCarveoutMaxShared;
#ifdef QG_TOOLS_KNOBS
    if (const char* v = std::getenv("QG_CARVEOUT")) carve = std::atoi(v);      // A/B runs: -1 = driver default, 0..100 = percent shared
#endif
    cudaError_t e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 32>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    if (e == cudaSuccess && smem_bytes > 48 * 1024) e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if constexpr (MODE == MODE_STEP) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 32, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        if (e == cudaSuccess && smem_bytes > 48 * 1024) e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 32, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    }
    if constexpr (MODE != MODE_OBSERVE) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 16>, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        if (e == cudaSuccess && smem_bytes > 48 * 1024) e = cudaFuncSetAttribute(k_step<KIND, MODE, INV, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    }
    return e;
}

template <int KIND>
cudaError_t prepare_step_kind(size_t smem_bytes) {
    cudaError_t e = prepare_one<KIND, MODE_STEP, 0>(smem_bytes);
    if (e == cudaSuccess) e = prepare_one<KIND, MODE_OBSERVE, 0>(smem_bytes);
    if (e == cudaSuccess) e = prepare_one<KIND, MODE_SEARCH, 0>(smem_bytes);
    if constexpr (kind_has_matrix_inverse(KIND)) {
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_STEP, 8>(smem_bytes);
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_STEP, 16>(smem_bytes);
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_STEP, 32>(smem_bytes);
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_SEARCH, 8>(smem_bytes);
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_SEARCH, 16>(smem_bytes);
        if (e == cudaSuccess) e = prepare_one<KIND, MODE_SEARCH, 32>(smem_bytes);
    }
    return e;
}

#define QG_INSTANTIATE_KIND(KIND)                                                                                              \
    template cudaError_t launch_step_kind<KIND>(int, int, const DevCfg&, const StepArgs&, const LaunchGeom&, cudaStream_t);    \
    template cudaError_t prepare_step_kind<KIND>(size_t);                                                                      \
    template cudaError_t launch_search_fused<KIND>(const DevCfg&, const StepArgs&, const PolicyDev&, int, int32_t*, size_t, long long*, const uint32_t*,            \
                                                   const SearchTwist*, cudaStream_t);                                                           \
    template cudaError_t search_fused_smem<KIND, false>(const PolicyDev&, size_t, int, size_t*, size_t*, size_t*);                             \
    template cudaError_t search_fused_smem<KIND, true>(const PolicyDev&, size_t, int, size_t*, size_t*, size_t*);

}  // namespace qg
