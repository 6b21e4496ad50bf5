// qg_policy.cu — the policy's action network evaluated straight from packed-bit observations (SURVEY.md §8f row 3).
//
// twisterl feeds Env::observe()'s sparse indices to an embedding-bag first layer (the reason observe() returns indices,
// e.g. clifford.rs:361-368); the dense f32 observation the engine materialises for a PyTorch policy is 32x larger than
// the information it carries.  Here the observation stays packed (one bit per entry, written by the step kernel) and the
// first layer is a gather-sum of weight columns over the set bits; the remaining layers of the BasicPolicy-shaped MLP
// (Linear -> ReLU chain, examples/models/*.pt) and the softmax run in the same kernel, so one synth-search decision is
// two launches (this one + the fused sample/step kernel) instead of a dozen library kernels.
//
// Decomposition: one CTA of 256 threads owns 8 batch rows.  Activations live in shared memory as [feature][row]
// (32 bytes per feature: every thread reads the same address, a broadcast); thread j owns output features j, j+256, ..
// and keeps one f32 accumulator per (feature, row) in registers, so each weight feeds 8 FMAs.  Weights are kept
// transposed ([in][out], rows padded to 16 bytes) and stream L2 -> shared memory in 16 KB tiles with cp.async.bulk
// completing on mbarriers, three tiles in flight, one flat tile schedule across all layers so the pipeline never
// drains at a layer boundary.  The first layer is an exact gather-sum in fixed point (layer0_fixed in qg_policy_kernels.cuh:
// 64-bit integer accumulators, order independent), which the one-launch search updates incrementally from the observation
// bits that changed; the dense layers sum over the input features in f32 FMA chains that split each weight tile's rows over 2, 4 or 16
// thread groups and combine them in a fixed order (include/qg_engine.h, qg_policy_create, states the order).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "qg_host.hpp"
#include "qg_policy_host.hpp"

namespace qg {

__global__ void __launch_bounds__(kPolThreads) k_policy_mlp(const __grid_constant__ PolicyDev p, const uint32_t* bits, int64_t B, float* probs, float* logits_out,
                                                            float* values_out) {
    extern __shared__ __align__(128) float sm[];
    const PolicySmem ps = policy_smem_carve(p, sm);
    policy_init_barriers(ps, threadIdx.x);
    // programmatic dependent launch: everything above overlaps the tail of the previous kernel in the stream (the step kernel that
    // writes `bits`); the next kernel (the step kernel that reads `probs`) may be scheduled now, it waits for this grid itself
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    __syncthreads();                               // barriers initialised
    int G = 0;
    policy_forward_rows(p, ps, bits, (int64_t)blockIdx.x * kPolRows, B, probs, logits_out, G, 0, -1, nullptr, nullptr, 0, values_out);
}

}  // namespace qg

using namespace qg;

#define POL_CUDA_OK(expr)                                                                      \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
            return QG_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

extern "C" {

void qg_policy_destroy(qg_policy* p) {
    if (!p) return;
    for (float* b : p->bufs) cudaFree(b);
    if (p->acc0) cudaFree(p->acc0);
    delete p;
}

int qg_policy_create(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features, const float* const* weights_host,
                     const float* const* biases_host, qg_policy** out) {
    return qg_policy_create_value(device, obs_size, num_layers, out_features, weights_host, biases_host, nullptr, 0.0f, out);
}

int qg_policy_create_value(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features, const float* const* weights_host,
                           const float* const* biases_host, const float* value_weight_host, float value_bias, qg_policy** out) {
    if (!out) { set_error("null out"); return QG_ERR_INVALID; }
    *out = nullptr;
    if (obs_size < 1 || obs_size > 65535) { set_error("qg_policy_create: obs_size must be in [1, 65535]"); return QG_ERR_UNSUPPORTED; }
    if (num_layers < 1 || num_layers > kPolMaxLayers || !out_features || !weights_host || !biases_host) { set_error("qg_policy_create: 1..8 layers with weights and biases"); return QG_ERR_INVALID; }
    int maxw = 0;
    const int extra = value_weight_host ? 1 : 0;            // the value head rides along as one more output of the last layer
    for (int l = 0; l < num_layers; ++l) {
        const int o = out_features ? out_features[l] + (l == num_layers - 1 ? extra : 0) : 0;
        if (out_features[l] < 1 || o > kPolMaxWidth) { set_error("qg_policy_create: layer widths must be in [1, 1024]"); return QG_ERR_UNSUPPORTED; }
        if (!weights_host[l] || !biases_host[l]) { set_error("qg_policy_create: null layer"); return QG_ERR_INVALID; }
        maxw = std::max(maxw, o);
    }
    int ndev = 0;
    POL_CUDA_OK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { set_error("no such CUDA device (the engine has no CPU fallback)"); return QG_ERR_CUDA; }
    POL_CUDA_OK(cudaSetDevice(device));
    qg_policy* p = new (std::nothrow) qg_policy();
    if (!p) { set_error("out of memory"); return QG_ERR_INVALID; }
    p->device = device;
    PolicyDev& d = p->d;
    d.num_layers = num_layers; d.obs_size = obs_size; d.obs_words = (obs_size + 31) / 32;
    d.act0_floats = maxw * kPolRows;
    d.act1_floats = maxw * kPolRows;
    for (int l = 0; l < num_layers; ++l) {
        const bool last = l == num_layers - 1;
        const int in = l == 0 ? obs_size : out_features[l - 1], o0 = out_features[l], o = o0 + (last ? extra : 0), os = (o + 3) / 4 * 4;
        d.width[l] = o; d.stride[l] = os;
        std::vector<float> t((size_t)in * os, 0.0f), bias(o, 0.0f);
        for (int j = 0; j < o0; ++j) for (int k = 0; k < in; ++k) t[(size_t)k * os + j] = weights_host[l][(size_t)j * in + k];   // torch Linear.weight is [out][in]
        std::memcpy(bias.data(), biases_host[l], (size_t)o0 * 4);
        if (last && extra) { for (int k = 0; k < in; ++k) t[(size_t)k * os + o0] = value_weight_host[k]; bias[o0] = value_bias; }
        if (l == 0) {
            // fixed point for the exact (order-independent) first-layer sum: the largest |weight| lands just below 2^30
            float mx = 0.0f;
            for (float v : t) { if (!std::isfinite(v)) { set_error("qg_policy_create: non-finite weight"); qg_policy_destroy(p); return QG_ERR_INVALID; } mx = std::max(mx, std::fabs(v)); }
            int shift = 30;
            if (mx > 0.0f) { int e = 0; std::frexp(mx, &e); shift = std::min(30 - e, 120); }      // mx < 2^e  =>  mx * 2^(30-e) < 2^30
            d.w0_scale = std::ldexp(1.0f, -shift);
            for (float& v : t) { const int32_t q = (int32_t)std::llrint(std::ldexp((double)v, shift)); std::memcpy(&v, &q, 4); }
        }
        float *w = nullptr, *b = nullptr;
        cudaError_t ce = cudaMalloc(&w, t.size() * 4);
        if (ce == cudaSuccess) { p->bufs.push_back(w); ce = cudaMalloc(&b, (size_t)o * 4); }
        if (ce == cudaSuccess) { p->bufs.push_back(b); ce = cudaMemcpy(w, t.data(), t.size() * 4, cudaMemcpyHostToDevice); }
        if (ce == cudaSuccess) ce = cudaMemcpy(b, bias.data(), (size_t)o * 4, cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) { set_error(std::string("qg_policy_create: ") + cudaGetErrorString(ce)); qg_policy_destroy(p); return QG_ERR_CUDA; }
        d.wt[l] = l == 0 ? nullptr : w; d.bias[l] = b;
        if (l == 0) d.w0q = reinterpret_cast<const int32_t*>(w);
    }
    d.num_actions = out_features[num_layers - 1];
    p->smem = policy_smem_bytes(d);
    if (p->smem > 210 * 1024) { set_error("qg_policy_create: the network needs more shared memory than one SM has"); qg_policy_destroy(p); return QG_ERR_UNSUPPORTED; }
    {
        cudaError_t ce = cudaFuncSetAttribute(k_policy_mlp, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
        if (ce == cudaSuccess && p->smem > 48 * 1024) ce = cudaFuncSetAttribute(k_policy_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
        if (ce != cudaSuccess) { set_error(std::string("qg_policy_create: ") + cudaGetErrorString(ce)); qg_policy_destroy(p); return QG_ERR_CUDA; }
    }
    *out = p;
    return QG_OK;
}

int32_t qg_policy_num_actions(const qg_policy* p) { return p ? p->d.num_actions : 0; }
int32_t qg_policy_has_value(const qg_policy* p) { return (p && p->d.width[p->d.num_layers - 1] > p->d.num_actions) ? 1 : 0; }

int qg_policy_forward_bits(qg_policy* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev, float* logits_dev, qg_stream stream) {
    return qg_policy_forward_bits_value(p, obs_bits_dev, batch, probs_dev, logits_dev, nullptr, stream);
}

int qg_policy_forward_bits_value(qg_policy* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev, float* logits_dev, float* values_dev,
                                 qg_stream stream) {
    if (!p || !obs_bits_dev || (!probs_dev && !logits_dev && !values_dev)) { set_error("null argument"); return QG_ERR_INVALID; }
    if (values_dev && !qg_policy_has_value(p)) { set_error("qg_policy_forward_bits_value: the policy was created without a value head"); return QG_ERR_INVALID; }
    if (batch < 0) { set_error("qg_policy_forward_bits: negative batch"); return QG_ERR_INVALID; }
    if (batch == 0) return QG_OK;
    int cur = -1;
    POL_CUDA_OK(cudaGetDevice(&cur));
    if (cur != p->device) POL_CUDA_OK(cudaSetDevice(p->device));
    const unsigned grid = (unsigned)((batch + kPolRows - 1) / kPolRows);
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(kPolThreads); lc.dynamicSmemBytes = p->smem; lc.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at; lc.numAttrs = 1;
    POL_CUDA_OK(cudaLaunchKernelEx(&lc, k_policy_mlp, p->d, obs_bits_dev, batch, probs_dev, logits_dev, values_dev));
    return QG_OK;
}

}  // extern "C"
