// qg_aux_kernels.cuh — small non-template kernels (record readers, best-rollout reduction); included by qg_engine.cu only.
#pragma once
#include "qg_kernels.cuh"

namespace qg {

// ---- small readers -----------------------------------------------------------------------------------
__global__ void k_read_status(const __grid_constant__ DevCfg c, float* reward, uint8_t* done, uint8_t* success, int32_t* depth) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= c.B) return;
    const uint32_t d = c.rec[(size_t)HD_DEPTH * c.Bpad + env], f = c.rec[(size_t)HD_FLAGS * c.Bpad + env];
    if (reward) reward[env] = __uint_as_float(c.rec[(size_t)HD_REWARD * c.Bpad + env]);
    if (done) done[env] = (d == 0 || (f & FL_SUCCESS)) ? 1 : 0;
    if (success) success[env] = (f & FL_SUCCESS) ? 1 : 0;
    if (depth) depth[env] = (int32_t)d;
}
__global__ void k_read_metrics(const __grid_constant__ DevCfg c, uint32_t* out) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= c.B) return;
    const uint32_t l = c.rec[(size_t)HD_LAYERS * c.Bpad + env];
    reinterpret_cast<uint4*>(out)[env] = make_uint4(c.rec[(size_t)HD_NCNOTS * c.Bpad + env], l >> 16, l & 0xFFFFu, c.rec[(size_t)HD_NGATES * c.Bpad + env]);
}
__global__ void k_read_errors(const __grid_constant__ DevCfg c, uint32_t* out) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= c.B) return;
    out[env] = (c.rec[(size_t)HD_FLAGS * c.Bpad + env] >> FL_ERR_SHIFT) & 0xFFu;
}
__global__ void k_fill_f32(float* p, int64_t n, float v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_copy_f32(const float* src, float* dst, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}

// ---- best-rollout reduction (synth search): arg-max of the packed key rollout_key (qg_kernels.cuh) ----------------------------------
__global__ void k_best(const __grid_constant__ DevCfg c, unsigned long long* best) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long key = 0;
    if (env < c.B) {
        const uint32_t f = c.rec[(size_t)HD_FLAGS * c.Bpad + env];
        key = rollout_key((f & FL_SUCCESS) != 0, c.ret[env], c.first_id + env);
    }
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o); key = other > key ? other : key; }
    if ((threadIdx.x & 31) == 0 && key) atomicMax(best, key);
}

// ---- rollout-collector helpers ------------------------------------------------------------------------
// Generalised advantage estimation over a [T][B] rollout, one thread per environment walking its column backwards
// (every load / store of a warp is one coalesced row segment).  Each product and sum is rounded on its own, in the
// order written, so the CPU restatement matches bit for bit:
//     nd      = done[t] ? 0 : 1
//     delta   = (reward[t] + (gamma * value[t+1]) * nd) - value[t]
//     adv[t]  = delta + ((gamma * lambda) * nd) * adv[t+1]          (adv[T] = 0)
//     ret[t]  = adv[t] + value[t]
// A step with valid[t] == 0 (the env was already final at decision time and was not stepped) yields adv = ret = 0 and
// cuts the recursion like an episode end.
__global__ void k_gae(const float* __restrict__ reward, const float* __restrict__ value, const uint8_t* __restrict__ done,
                      const uint8_t* __restrict__ valid, int T, int64_t B, float gamma, float lambda, float* __restrict__ adv, float* __restrict__ ret) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float gl = __fmul_rn(gamma, lambda);
    float next_v = value[(size_t)T * B + b], next_adv = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
        const size_t k = (size_t)t * B + b;
        const float v = value[k];
        if (valid && !valid[k]) { adv[k] = 0.0f; if (ret) ret[k] = 0.0f; next_adv = 0.0f; next_v = v; continue; }
        const float nd = done[k] ? 0.0f : 1.0f;
        const float delta = __fsub_rn(__fadd_rn(reward[k], __fmul_rn(__fmul_rn(gamma, next_v), nd)), v);
        const float a = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nd), next_adv));
        adv[k] = a;
        if (ret) ret[k] = __fadd_rn(a, v);
        next_adv = a; next_v = v;
    }
}

// Twists (symmetry.rs:297-361) applied on the device: out[b][j] = in[b][table[k[b]][j]] for a [K][len] index table.
// With the inverse of obs_perms it produces the twisted observation (index i of the observation moves to
// obs_perms[k][i]); with act_perms it maps the policy's action weights back to the environment's action order.
__global__ void k_twist_gather(const float* __restrict__ in, float* __restrict__ out, const int32_t* __restrict__ table,
                               const int32_t* __restrict__ kidx, int64_t B, int len, uint64_t magic_len) {
    const int64_t total = B * (int64_t)len;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = magic_len ? (int64_t)__umul64hi((uint64_t)i, magic_len) : i;   // magic_len = ceil(2^64 / len), 0 for len == 1
        const int j = (int)(i - b * len);
        const int32_t k = kidx ? kidx[b] : 0;
        out[i] = in[b * len + table[(size_t)k * len + j]];
    }
}

// Twists on packed observations (qg_twist_bits): twist_word (qg_common.cuh) with qpinv[k] = p^-1 of twist k — qg_twist_gather with the
// inverse obs perm, on bits, from a [K][n] byte table instead of a [K][d*d] index table.
// Thread = (env, output word).  Twist index: kidx_in[b], or drawn  mulhi(philox(*seed_dev, first + b, draw, STREAM_TWIST), K)  (the seed
// is read at run time, so the launch can live in a CUDA graph); written to kidx_out[b] when given.
__global__ void k_twist_bits(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int ow, int obs_size, int n, int d,
                             const uint8_t* __restrict__ qpinv, uint32_t K, const int32_t* __restrict__ kidx_in, const uint64_t* __restrict__ seed_dev,
                             int64_t first, uint32_t draw, int32_t* __restrict__ kidx_out, int64_t B) {
    const int64_t total = B * (int64_t)ow;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / ow;
        const int w = (int)(i - b * ow);
        const uint32_t k = kidx_in ? (uint32_t)kidx_in[b] : __umulhi(philox_draw(*seed_dev, (uint64_t)(first + b), draw, STREAM_TWIST), K);
        if (kidx_out && w == 0) kidx_out[b] = (int32_t)k;
        const uint32_t* const row = in + (size_t)b * ow;
        out[i] = twist_word([&](int s) { return (__ldg(row + (s >> 5)) >> (s & 31)) & 1u; }, w, obs_size, n, d, qpinv + (size_t)k * n);
    }
}

// The twisted search's observation (qg_search_observe_twisted, qg_search_step_twisted): the packed observation of every rollout in the
// frame of its next decision, k = twist_draw(seed, first_id + b, HD_TICK), read straight from the records (record_twist_word); k goes to
// twist[b].  Thread = (rollout, output word).
template <int KIND>
__global__ void k_observe_twisted(const __grid_constant__ DevCfg c, uint32_t* __restrict__ out, int ow, const uint8_t* __restrict__ qpinv, uint32_t K, int d,
                                  int32_t* __restrict__ twist) {
    const int64_t total = c.B * (int64_t)ow;
    const int n = c.n;
    const uint64_t seed = seed_of(c);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / ow;
        const int w = (int)(i - b * ow);
        const uint32_t k = twist_draw(seed, c.first_id + b, c.rec[(size_t)HD_TICK * c.Bpad + b], K);
        if (w == 0) twist[b] = (int32_t)k;
        const uint32_t* const st = c.rec + (size_t)c.off_state * c.Bpad + b;         // state word v of rollout b at st[v * Bpad]
        out[i] = record_twist_word<KIND>(st, c.Bpad, w, c.obs_size, n, d, qpinv + (size_t)k * n);
    }
}

}  // namespace qg
