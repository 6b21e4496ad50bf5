// qg_common.cuh — record layout, device config and bit helpers shared by the engine kernels.
//
// HBM layout (structure of arrays, "word planes"): every environment owns W 32-bit words; word w of
// environment e lives at rec[w * Bpad + e] (Bpad = batch rounded up to 32), so a warp that handles 32
// consecutive environments moves each word plane with one fully coalesced 128-byte transaction.
//
//   words 0..6   header   depth | flags | n_cnots | n_gates | layers | reward | tick
//   then         last_gates[n]  (int16 pairs, -1 = 0xFFFF)      metrics.rs:24
//   then         last_cxs[n]    (int16 pairs)                   metrics.rs:25
//   then         state          kind specific, bit packed (see below)
//   then         PauliNetwork extras (phase planes, alive mask, DAG node order, anticommutation rows)
//
// state encodings
//   Permutation     n bytes, 4 per word                               (permutation.rs:30  Vec<usize>)
//   LinearFunction  dense bit stream, entry (r,c) at bit r*n+c         (linear_function.rs:29-33, one byte per bit there)
//   Clifford        dense bit stream, entry (r,c) at bit r*2n+c        (clifford.rs:28-31)
//   PauliNetwork    2n rows of CW bits, CW = 2n+Rtot rounded up to whole words (a row operation is one word
//                   operation per row word); columns 2n.. hold the rotations' (x|z) vectors, which keep evolving
//                   after a rotation is harvested exactly like PauliNetwork::rotation_qk does
//                   (pauli_network.rs:189-223); `alive` masks them.
// For LinearFunction/Clifford the state bit stream IS the observation bit stream (observe() lists the
// set bits in row-major order, clifford.rs:361-368), so the observation expander reads it directly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/qg_engine.h"

namespace qg {

// header word indices
enum { HD_DEPTH = 0, HD_FLAGS = 1, HD_NCNOTS = 2, HD_NGATES = 3, HD_LAYERS = 4, HD_REWARD = 5, HD_TICK = 6, HD_WORDS = 7 };
// flags word: bit0 success, bit1 inverted, bits 8..15 error flags (QG_FLAG_*), bits 16..31 solution length
enum { FL_SUCCESS = 1u, FL_INVERTED = 2u, FL_ERR_SHIFT = 8, FL_LEN_SHIFT = 16 };
// PauliNetwork extra words (relative to off_extra)
enum { PX_PLO = 0, PX_PHI = 1, PX_ALIVE = 2, PX_ORD0 = 3, PX_ORD1 = 4, PX_MISC = 5, PX_ANTI = 6 };
// PX_MISC: bits 0..15 current_perm_idx, bits 16..23 rotations loaded (R), bits 24..31 live DAG nodes (m)

// Philox stream ids (1..4 shared with oracle/qg_oracle.hpp; STREAM_TWIST: the collector's per-env twist pick, qg_twist_bits)
enum : uint32_t { STREAM_RESET = 1, STREAM_COIN = 2, STREAM_PERM = 3, STREAM_SAMPLE = 4, STREAM_TWIST = 5 };

constexpr int kThreads = 256;          // threads per CTA of the step kernels
constexpr int kMaxRot = 16;            // rotations per PauliNetwork env (nibble-coded DAG order)

struct DevCfg {
    int32_t kind, n, D, A, obs_size, obs_cols;
    int32_t SW, MW, W, off_lastg, off_lastcx, off_state, off_extra, OW;   // word counts / offsets
    int32_t max_depth, depth_slope, difficulty, add_inverts, track, sol_cap;
    int32_t max_rot, Rtot, CW, nperms;
    float w0, w1, w2, w3, plr;
    int64_t B, Bpad;
    uint32_t* rec;            // [W][Bpad]
    uint32_t* sol;            // [sol_cap][Bpad]
    float* ret;               // [Bpad] search returns
    const uint32_t* gates;    // [A] kind | q0<<8 | q1<<16
    const uint32_t* ident;    // [SW] identity state (LF/Clifford) — solved() target
    const uint8_t* qperms;    // [nperms][n]   PauliNetwork qubit permutations (pauli.rs:289-290)
    const uint16_t* aperms;   // [nperms][A]
    const uint32_t* pgen;     // PauliNetwork reset generator tables (see k_reset_pauli)
    uint64_t seed; int64_t first_id;
    const uint64_t* seed_dev; // if set, the Philox seed is read from device memory at launch time instead (CUDA-graph replays: the host
                              // rewrites the word between replays; qg_reset_select_dev / qg_collect_step_dev)
    uint32_t magic_n;         // ceil(2^32 / n): exact division of obs offsets by n (Permutation expander)
    int32_t row_shift;        // LinearFunction / Clifford: log2(D) when D is a power of two <= 32 (a row then lies inside one word at bit offset
                              // (r << row_shift) & 31 and the row primitives are one load / shift / xor / store), else -1
};

// ---- Philox4x32-10: key = seed, counter = (env lo, env hi, draw index, stream) ----------------
__host__ __device__ __forceinline__ uint32_t philox_draw(uint64_t seed, uint64_t env, uint32_t idx, uint32_t stream) {
    uint32_t c0 = (uint32_t)env, c1 = (uint32_t)(env >> 32), c2 = idx, c3 = stream;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t seed_of(const DevCfg& c) { return c.seed_dev ? *c.seed_dev : c.seed; }
// ---- per-thread word array living in shared memory with stride EPC (bank == lane, conflict free
//      for any per-thread dynamic index) ------------------------------------------------------------
template <int EPC>
struct SmWords {
    uint32_t* p;
    __device__ __forceinline__ uint32_t& operator[](int i) const { return p[i * EPC]; }
    __device__ __forceinline__ SmWords at(int i) const { return SmWords{p + i * EPC}; }
};

// bits [o, o+len) of a dense bit stream, len in 1..32
template <class Wd>
__device__ __forceinline__ uint32_t get_bits(const Wd& W, int o, int len) {
    const int w = o >> 5, s = o & 31;
    const uint32_t lo = W[w];
    const uint32_t hi = (s + len > 32) ? W[w + 1] : 0u;
    const uint32_t v = __funnelshift_r(lo, hi, s);
    return len >= 32 ? v : (v & ((1u << len) - 1u));
}
// stream[o, o+len) ^= v   (v has no bits above len)
template <class Wd>
__device__ __forceinline__ void xor_bits(const Wd& W, int o, int len, uint32_t v) {
    const int w = o >> 5, s = o & 31;
    W[w] ^= v << s;
    if (s + len > 32) W[w + 1] ^= v >> (32 - s);
}
template <class Wd>
__device__ __forceinline__ uint32_t get_bit(const Wd& W, int o) { return (W[o >> 5] >> (o & 31)) & 1u; }

// row primitives on a dense bit matrix whose rows are `rb` bits wide
// ... rows that never straddle a word (rb = 1 << sh <= 32): the warp-uniform fast path of the LinearFunction / Clifford gates
template <class Wd>
__device__ __forceinline__ uint32_t row_get_pow2(const Wd& W, int sh, int r) {
    const int o = r << sh;
    const uint32_t v = W[o >> 5] >> (o & 31);
    return sh == 5 ? v : (v & ((1u << (1 << sh)) - 1u));
}
template <class Wd>
__device__ __forceinline__ void row_xor_pow2(const Wd& W, int sh, int dst, int src) {
    const int o = dst << sh;
    W[o >> 5] ^= row_get_pow2(W, sh, src) << (o & 31);
}
template <class Wd>
__device__ __forceinline__ void row_swap_pow2(const Wd& W, int sh, int a, int b) {
    const uint32_t d = row_get_pow2(W, sh, a) ^ row_get_pow2(W, sh, b);
    const int oa = a << sh, ob = b << sh;
    W[oa >> 5] ^= d << (oa & 31);
    W[ob >> 5] ^= d << (ob & 31);              // (after the first store: a and b may share a word)
}
template <class Wd>
__device__ __forceinline__ void row_xor(const Wd& W, int rb, int dst, int src) {   // row dst ^= row src (dst==src zeroes it)
    for (int c0 = 0; c0 < rb; c0 += 32) {
        const int len = min(32, rb - c0);
        xor_bits(W, dst * rb + c0, len, get_bits(W, src * rb + c0, len));
    }
}
template <class Wd>
__device__ __forceinline__ void row_swap(const Wd& W, int rb, int a, int b) {
    for (int c0 = 0; c0 < rb; c0 += 32) {
        const int len = min(32, rb - c0);
        const uint32_t d = get_bits(W, a * rb + c0, len) ^ get_bits(W, b * rb + c0, len);
        xor_bits(W, a * rb + c0, len, d);
        xor_bits(W, b * rb + c0, len, d);
    }
}
// int16 pairs (last_gates / last_cxs)
template <class Wd>
__device__ __forceinline__ int get16(const Wd& W, int q) { return (int)(int16_t)(W[q >> 1] >> ((q & 1) * 16)); }
template <class Wd>
__device__ __forceinline__ void set16(const Wd& W, int q, int v) {
    const int s = (q & 1) * 16;
    W[q >> 1] = (W[q >> 1] & ~(0xFFFFu << s)) | (((uint32_t)v & 0xFFFFu) << s);
}
// bytes (permutation entries)
template <class Wd>
__device__ __forceinline__ uint32_t get8(const Wd& W, int i) { return (W[i >> 2] >> ((i & 3) * 8)) & 0xFFu; }
template <class Wd>
__device__ __forceinline__ void set8(const Wd& W, int i, uint32_t v) {
    const int s = (i & 3) * 8;
    W[i >> 2] = (W[i >> 2] & ~(0xFFu << s)) | ((v & 0xFFu) << s);
}
#endif  // __CUDACC__

}  // namespace qg
