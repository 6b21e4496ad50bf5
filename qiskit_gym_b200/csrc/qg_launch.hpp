// qg_launch.hpp — host-side launch interface of the fused step kernel.  Each environment kind is compiled in its own
// translation unit (qg_step_<kind>.cu) so the template instantiations build in parallel.
#pragma once
#include <cuda_runtime.h>

#include "qg_kernels.cuh"

namespace qg {

struct LaunchGeom {
    unsigned grid;
    size_t smem_bytes;
    int pdl;            // launch with the programmatic-stream-serialization attribute
    int epw = 32;       // environments per warp tile: 32 or 16 (see step_tile)
    const void* l2_base = nullptr;   // persisting-L2 access window (bytes 0 = none)
    size_t l2_bytes = 0;
};

// mode: MODE_STEP / MODE_OBSERVE / MODE_SEARCH;  inv: 0 / 8 / 16 / 32 (see k_step)
template <int KIND>
cudaError_t launch_step_kind(int mode, int inv, const DevCfg& c, const StepArgs& a, const LaunchGeom& g, cudaStream_t st);
// opt in to > 48 KB dynamic shared memory for every instantiation of the kind (outside any stream capture)
template <int KIND>
cudaError_t prepare_step_kind(size_t smem_bytes);

// the whole rollout search in one launch (qg_search_fused.cuh); step_smem_bytes = one warp region of the step kernel; tw: the twisted
// search's tables, or null
struct PolicyDev;
// The twisted search's tables (k_search_fused<KIND, true>; the launch's a.act_perm holds the [K][A] act perms and a.twist = twist).
struct SearchTwist {
    const uint8_t* qpinv;        // [K][n] inverse qubit permutation of every twist (collector.qubit_twist_table)
    int32_t* twist;              // [B] the frame of each rollout's current decision
    uint32_t K;
    int32_t d;                   // side of the square observation: n (Permutation, LinearFunction) or 2n (Clifford)
};
template <int KIND>
cudaError_t launch_search_fused(const DevCfg& c, const StepArgs& a, const PolicyDev& p, int max_decisions, int32_t* decisions_out, size_t step_smem_bytes, long long* acc0, const uint32_t* first_bits,
                                const SearchTwist* tw, cudaStream_t st);
// the shared memory a launch_search_fused CTA needs (the dynamic bytes it requests, the kernel's static bytes) and the most one block
// may have on `device`
template <int KIND, bool TWIST>
cudaError_t search_fused_smem(const PolicyDev& p, size_t step_smem_bytes, int device, size_t* dynamic_bytes, size_t* static_bytes, size_t* limit);

}  // namespace qg
