// qg_kernels.cuh — the fused environment kernels (sm_100a).
//
// One launch of k_step does, for every environment of the batch, what the reference does with five
// trait calls per environment (step, reward, is_final, observe, masks — e.g. clifford.rs:321-368):
//   phase 1 (one thread per environment, state staged in shared memory):
//       gate lookup -> MetricsTracker update (metrics.rs:64-123) -> weighted penalty (metrics.rs:135-146)
//       -> gate applied as row XOR / row swap on the packed GF(2) state -> solution log -> depth tick
//       -> optional inverse (coin) -> solved() -> reward -> write-back;
//   phase 2 (the whole warp, for its 32 environments): the contiguous slab of the dense float observation tensor and
//       of the uint8 action-mask tensor is produced from the packed bits with 16-byte coalesced streaming stores.
#pragma once
#include <type_traits>

#include "qg_common.cuh"
#include "qg_gf2.cuh"

namespace qg {

struct StepArgs {
    const int32_t* actions;      // [B]            (MODE_STEP)
    const uint8_t* actions8;     // [B] or null: the same stream as one byte per action (the packed host wire format, num_actions <= 256); read instead of `actions`
    uint32_t* done_bits;         // [ceil(B/32)][bits_stride] or null: is_final of tile k (envs 32k..32k+31, bit = env % 32) after step t at [k][bits_t0 + t] ...
    uint32_t* success_bits;      // ... and success, same layout: 2 bits per env-step instead of two bytes, written as whole 128-byte lines every 32 steps
    int32_t bits_stride, bits_t0;
    const uint8_t* coins;        // [B] or null
    const uint32_t* perm_raw;    // [B] or null
    const float* weights;        // [B][A]         (MODE_SEARCH)
    int32_t deterministic;
    float* obs;                  // [B][obs_size] or null
    uint32_t* obs_bits;          // [B][ceil(obs_size/32)] or null: the observation as packed bits (bit i of an env = entry i), env-major
    const int32_t* src_slot;     // [B] or null: logical env i reads its record from record slot src_slot[i] ...
    const int32_t* dst_slot;     // [B] or null: ... and writes it to slot dst_slot[i] (clone + step in one pass: tree search nodes)
    int32_t skip_negative;       // MODE_STEP: a negative action leaves the env untouched (no step, no outputs) instead of flagging it
    uint8_t* mask;               // [B][A] or null
    float* reward; uint8_t* done; uint8_t* success;   // [B] or null
    int32_t* chosen;             // [B] or null    (MODE_SEARCH)
    const int32_t* act_perm;     // [K][A] or null (MODE_SEARCH, twisted collector): `weights` are in the policy's (twisted) action order and env
    const int32_t* twist;        // [B]              action g reads weights[act_perm[twist[env]][g]]  (qg_collect_step_twisted_dev)
    int32_t* policy_chosen;      // [B] or null    (MODE_SEARCH) the chosen action in the weights' order, act_perm[twist[env]][chosen]; -1: not stepped
    int32_t* num_active;         // [1] or null    (MODE_SEARCH)
    int32_t nsteps;              // steps played by this launch (MODE_STEP; 1 otherwise)
    int32_t ring;                // obs / mask hold `ring` step slots of [B][obs_size] / [B][A]; step t writes slot (slot0 + t) % ring
    int32_t slot0;
    int32_t symplectic;          // Clifford: every loaded state is symplectic, the coin's inverse may use J M^T J (qg_gf2.cuh)
    int32_t pdl_mode;            // 0: plain launch; 1: dependents may launch right away; 2: only once this grid owns the records
    int32_t stagger_ns, num_sms; // replay: warp k of an SM starts k * stagger_ns late so that the warps of an SM do not all
                                 // alternate between the latency-bound step phase and the store-bound expansion in lock-step
    int64_t in_stride;           // elements between consecutive steps of actions / coins / perm_raw
    int64_t out_stride;          // elements between consecutive steps of reward / done / success
    int32_t sm_warp_words, sm_scr, sm_obs;   // per-warp shared-memory region size and sub-region offsets (words)
    int32_t sm_cat;                          // offset of the tile's concatenated observation bit stream (expand_cat), or -1: not used by this launch
    int32_t sm_wts;                          // MODE_SEARCH: offset of the tile's staged action weights [env][A | 1], or -1: read them from global memory
    const uint32_t* in_flags;                // replay from a staging buffer the copy engine is still filling (qg_replay_host_packed): in_flags[k] != 0 once the
    int32_t in_chunk[4];                     // action / coin rows from step in_chunk[k] on have arrived (-1: no such chunk); null: all resident
    int32_t pair;                            // replay with a warp PAIR per tile: warp 0 plays the steps, warp 1 expands / stores the observations (step_tile)
    int32_t sm_pair, pair_words;             // offset of the pair's two hand-over buffers ([2][pair_words] words, then 2 header words) in the tile's region
    int32_t sm_pair_bar;                     // offset (words, 8-byte aligned) of four mbarriers (QG_PAIR_MBARRIER tools builds only; the product uses named barriers)
    uint64_t magic_obs, magic_A;      // ceil(2^40/obs_size), ceil(2^40/A)   (general paths)
    uint64_t magic_ow;                // ceil(2^40/ceil(obs_size/32))        (packed observation)
    uint32_t magic_vpe, magic_a4;     // ceil(2^32/(obs_size/4)), ceil(2^32/(A/4))   (fast paths)
    uint32_t exp_q, exp_r;            // 32 / VPE and 32 % VPE with VPE = obs_size / 4: how (env, float4-in-env) advances per warp store
};

enum { MODE_STEP = 0, MODE_OBSERVE = 1, MODE_SEARCH = 2 };

__device__ __forceinline__ uint32_t fastdiv40(uint32_t x, uint64_t magic) { return (uint32_t)(((uint64_t)x * magic) >> 40); }

struct Counts { uint32_t nc, ng, nl, nlc; };

// MetricsTracker::apply_gate (metrics.rs:64-123) in closed form, one select-based routine for every gate kind so that a warp
// whose lanes hold different gates runs it once.  The reference expands  CX -> cx(c,t);  SWAP -> cx(c,t), cx(t,c), cx(c,t);
// CZ -> single(t), cx(c,t), single(t);  one-qubit gate -> single(q)  (77-80), with
//   single(t): n_gates++, L = last_gates[t]+1 -> last_gates[t], layers                                  (84-96)
//   cx(c,t)  : ignored if c == t; n_cnots++, n_gates++, L = max(last_gates[c], last_gates[t])+1 -> both, same on last_cxs (98-123)
// k chained cx on the same pair raise both qubits to max+k, so the whole gate is
//   [pre single on t] -> [cx raising by k] -> [post single on t]   with (pre, k, post) = 1q (1,0,0), CX (0,1,0), SWAP (0,3,0), CZ (1,1,1).
// `layers` is always {0..max} (tests/test_oracle.py::test_layer_sets_are_prefixes), so len() is the running maximum + 1; the
// last value written to t is the largest of the chain.  Counters saturate at 32767 with a flag, stage by stage like the
// one-by-one updates would.
template <class Wd>
__device__ __forceinline__ void met_gate(const Wd& lg, const Wd& lc, int n, int kind, int q0, int q1, Counts& c, uint32_t& err) {
    (void)n;                                              // qubit indices were range-checked at construction (qg_config_validate)
    const bool two = kind >= QG_CX;
    const int t = two ? q1 : q0;
    const int pre = (!two || kind == QG_CZ) ? 1 : 0, post = (kind == QG_CZ) ? 1 : 0;
    const int k = (two && q0 != q1) ? (kind == QG_SWAP ? 3 : 1) : 0;
    auto sat = [&](int v) { if (v > 32767) { v = 32767; err |= QG_FLAG_LAYER_OVERFLOW; } return v; };
    int lt = sat(get16(lg, t) + pre);
    if (k) {
        lt = sat(max(get16(lg, q0), lt) + k);
        set16(lg, q0, lt);
        const int Lc = sat(max(get16(lc, q0), get16(lc, t)) + k);
        set16(lc, q0, Lc); set16(lc, t, Lc);
        c.nlc = max(c.nlc, (uint32_t)(Lc + 1));
        c.nc += (uint32_t)k;
    }
    lt = sat(lt + post);
    set16(lg, t, lt);
    c.nl = max(c.nl, (uint32_t)(lt + 1));
    c.ng += (uint32_t)(pre + k + post);
}
// metrics.rs:135-146: ((w0*dc + w1*dlc) + w2*dl) + w3*dg, every product and sum rounded on its own.
__device__ __forceinline__ float weighted_delta(const DevCfg& c, const Counts& now, const Counts& prev) {
    const float dc = (float)(now.nc - prev.nc), dlc = (float)(now.nlc - prev.nlc);
    const float dl = (float)(now.nl - prev.nl), dg = (float)(now.ng - prev.ng);
    float s = __fadd_rn(__fmul_rn(c.w0, dc), __fmul_rn(c.w1, dlc));
    s = __fadd_rn(s, __fmul_rn(c.w2, dl));
    s = __fadd_rn(s, __fmul_rn(c.w3, dg));
    return s;
}

// ---- state transitions ---------------------------------------------------------------------------
// permutation.rs:205-208 | linear_function.rs:237-243 + 62-83 | clifford.rs:249-260 + 89-133
template <int KIND, class Wd>
__device__ __forceinline__ void apply_gate_state(const DevCfg& c, const Wd& S, int kind, int q0, int q1) {
    if (KIND == QG_ENV_PERMUTATION) {
        if (kind == QG_SWAP) { const uint32_t a = get8(S, q0), b = get8(S, q1); set8(S, q0, b); set8(S, q1, a); }
    } else if (KIND == QG_ENV_LINEAR_FUNCTION) {
        if (q0 == q1) return;
        if (c.row_shift >= 0) {
            if (kind == QG_CX) row_xor_pow2(S, c.row_shift, q1, q0);
            else if (kind == QG_SWAP) row_swap_pow2(S, c.row_shift, q0, q1);
            return;
        }
        if (kind == QG_CX) row_xor(S, c.D, q1, q0);
        else if (kind == QG_SWAP) row_swap(S, c.D, q0, q1);
    } else if (KIND == QG_ENV_CLIFFORD) {
        const int n = c.n, D = c.D;
        // every gate is at most two row operations  A ^= B  or  A <-> B  on disjoint row pairs; written with selects so that a warp
        // whose lanes hold different gate kinds runs ONE routine instead of one switch arm per kind:
        //   H: q <-> n+q        S/Sdg: n+q ^= q        SX/SXdg: q ^= n+q
        //   CX: t ^= c, n+c ^= n+t        CZ: n+a ^= b, n+b ^= a        SWAP: a <-> b, n+a <-> n+b
        const bool two = kind >= QG_CX, swp = kind == QG_H || kind == QG_SWAP, en = !two || q0 != q1;
        const bool sx = kind == QG_SX || kind == QG_SXDG;
        int A0, B0, A1, B1;
        if (!two) { A0 = (kind == QG_H || sx) ? q0 : n + q0; B0 = (kind == QG_H || sx) ? n + q0 : q0; A1 = B1 = 0; }
        else if (kind == QG_CX) { A0 = q1; B0 = q0; A1 = n + q0; B1 = n + q1; }
        else if (kind == QG_CZ) { A0 = n + q0; B0 = q1; A1 = n + q1; B1 = q0; }
        else { A0 = q0; B0 = q1; A1 = n + q0; B1 = n + q1; }
        if (c.row_shift >= 0) {
            const int sh = c.row_shift;
            const uint32_t ra0 = row_get_pow2(S, sh, A0), rb0 = row_get_pow2(S, sh, B0);
            const uint32_t ra1 = row_get_pow2(S, sh, A1), rb1 = row_get_pow2(S, sh, B1);
            const uint32_t d0 = ra0 ^ rb0, d1 = ra1 ^ rb1;
            const uint32_t xa0 = en ? (swp ? d0 : rb0) : 0u, xb0 = (en && swp) ? d0 : 0u;
            const uint32_t xa1 = (en && two) ? (swp ? d1 : rb1) : 0u, xb1 = (en && two && swp) ? d1 : 0u;
            { const int o = A0 << sh; S[o >> 5] ^= xa0 << (o & 31); }
            { const int o = B0 << sh; S[o >> 5] ^= xb0 << (o & 31); }
            { const int o = A1 << sh; S[o >> 5] ^= xa1 << (o & 31); }
            { const int o = B1 << sh; S[o >> 5] ^= xb1 << (o & 31); }
            return;
        }
        // rows of any width (they may straddle words): the same two operations, 32 bits of a row at a time
        auto row_op = [&](int A, int B, bool on) {
            for (int c0 = 0; c0 < D; c0 += 32) {
                const int len = min(32, D - c0);
                const uint32_t rb = get_bits(S, B * D + c0, len), d = get_bits(S, A * D + c0, len) ^ rb;
                xor_bits(S, A * D + c0, len, on ? (swp ? d : rb) : 0u);
                xor_bits(S, B * D + c0, len, (on && swp) ? d : 0u);
            }
        };
        row_op(A0, B0, en);
        row_op(A1, B1, en && two);
    }
}

// solved(): permutation.rs:122-128 | linear_function.rs:91-100 | clifford.rs:136-145
template <int KIND, class Wd>
__device__ __forceinline__ bool solved_state(const DevCfg& c, const Wd& S) {
    if (KIND == QG_ENV_PERMUTATION) {
        for (int i = 0; i < c.n; ++i) if (get8(S, i) != (uint32_t)i) return false;
        return true;
    } else {
        if (S[0] != __ldg(c.ident)) return false;          // the usual case ends here (a scrambled state rarely shares its first word with the identity)
        uint32_t diff = 0;
        for (int w = 1; w < c.SW; ++w) diff |= S[w] ^ __ldg(c.ident + w);
        return diff == 0;
    }
}

// Gauss-Jordan inverse over GF(2) (linear_function.rs:124-146, clifford.rs:147-170); M, I: scratch bit streams.
template <class Wd>
__device__ bool invert_matrix(const DevCfg& c, const Wd& S, const Wd& M, const Wd& I) {
    const int D = c.D;
    for (int w = 0; w < c.SW; ++w) { M[w] = S[w]; I[w] = __ldg(c.ident + w); }
    for (int col = 0; col < D; ++col) {
        if (!get_bit(M, col * D + col)) {
            int pivot = -1;
            for (int r = col + 1; r < D; ++r) if (get_bit(M, r * D + col)) { pivot = r; break; }
            if (pivot < 0) return false;
            row_swap(M, D, col, pivot); row_swap(I, D, col, pivot);
        }
        for (int r = 0; r < D; ++r)
            if (r != col && get_bit(M, r * D + col)) { row_xor(M, D, r, col); row_xor(I, D, r, col); }
    }
    for (int w = 0; w < c.SW; ++w) S[w] = I[w];
    return true;
}
// permutation.rs:101-107
template <class Wd>
__device__ void invert_perm(const DevCfg& c, const Wd& S, const Wd& T) {
    for (int w = 0; w < c.SW; ++w) T[w] = 0;
    for (int i = 0; i < c.n; ++i) set8(T, (int)get8(S, i), (uint32_t)i);
    for (int w = 0; w < c.SW; ++w) S[w] = T[w];
}

// ---- PauliNetwork ----------------------------------------------------------------------------------
// Rows of the 2n x (2n + Rtot) matrix are padded to whole 32-bit words (c.CW = row stride in bits, a multiple of 32), so a
// row operation is one load / xor / store per row word, and the rotation part of a row (columns 2n .. 2n+Rtot) is one
// shifted word (two when it straddles a word, which depends on the configuration only: warp-uniform).
struct PauliRegs { uint32_t plo, phi, alive, ord0, ord1, misc; };
__device__ __forceinline__ uint32_t ord_get(const PauliRegs& p, int i) { return ((i < 8 ? p.ord0 : p.ord1) >> ((i & 7) * 4)) & 0xFu; }
__device__ __forceinline__ void ord_set(PauliRegs& p, int i, uint32_t v) {
    const int s = (i & 7) * 4;
    if (i < 8) p.ord0 = (p.ord0 & ~(0xFu << s)) | (v << s); else p.ord1 = (p.ord1 & ~(0xFu << s)) | (v << s);
}
__device__ __forceinline__ void phase_add(PauliRegs& p, uint32_t m) { const uint32_t carry = p.plo & m; p.plo ^= m; p.phi ^= carry; }
template <class Wd>
__device__ __forceinline__ uint32_t rot_bits(const DevCfg& c, const Wd& S, int row) {
    const int D = 2 * c.n, idx = row * (c.CW >> 5) + (D >> 5), sh = D & 31;
    uint32_t v = S[idx] >> sh;
    if (sh + c.Rtot > 32) v |= S[idx + 1] << (32 - sh);
    return c.Rtot >= 32 ? v : (v & ((1u << c.Rtot) - 1u));
}
template <class Wd>
__device__ __forceinline__ void pn_row_xor(const DevCfg& c, const Wd& S, int dst, int src) {
    const int RW = c.CW >> 5;
    for (int w = 0; w < RW; ++w) S[dst * RW + w] ^= S[src * RW + w];
}

// One-qubit gates as one routine with selects instead of branches, so that a warp whose lanes hold different gates runs it
// once: H (pauli_network.rs:189-194, pauli.rs:83-90): swap rows i, n+i, phase += 2(x & z);  S / Sdg = S^3 (209-215, 229-233;
// pauli.rs:92-97): row n+i ^= row i, phase += x or 3x;  SX / SXdg = SX^3 (217-223, 235-241; pauli.rs:105-110: H,S,H adds
// 2xz + z + 2z(1-x) = 3z, and 9z = z): row i ^= row n+i, phase += 3z or z.
__device__ __forceinline__ int pn_type_1q(int kind) { return kind + 1; }      // QG_H..QG_SXDG -> 1..5, 0 = none
template <class Wd>
__device__ __forceinline__ void pn_1q(const DevCfg& c, const Wd& S, PauliRegs& p, int type, int i) {
    const bool isH = type == 1, isS = type == 2 || type == 3, isSX = type == 4 || type == 5;
    const uint32_t x = rot_bits(c, S, i), z = rot_bits(c, S, c.n + i);
    phase_add(p, isS ? x : (isSX ? z : 0u));
    p.phi ^= isH ? (x & z) : (type == 3 ? x : (type == 4 ? z : 0u));
    const int RW = c.CW >> 5;
    for (int w = 0; w < RW; ++w) {
        const uint32_t a = S[i * RW + w], b = S[(c.n + i) * RW + w];
        S[i * RW + w] = isH ? b : (isSX ? (a ^ b) : a);
        S[(c.n + i) * RW + w] = isH ? a : (isS ? (a ^ b) : b);
    }
}
// pauli_network.rs:139-165 with the petgraph 0.6.5 retain_nodes/swap-remove node order (DESIGN.md §oracle).
// Harvested (axis, qubit, idx) triples are appended to hv[] as axis<<21 | qubit<<11 | idx<<1.
template <class Wd>
__device__ void pn_clean(const DevCfg& c, const Wd& S, const Wd& X, PauliRegs& p, const Wd& hv, int& nh, uint32_t& err) {
    const int n = c.n;
    for (;;) {
        int m = (int)(p.misc >> 24);
        if (m == 0) return;
        uint32_t ones = 0, ge2 = 0;                 // per-rotation weight of (x|z): bit-sliced saturating count
        for (int q = 0; q < n; ++q) { const uint32_t mk = rot_bits(c, S, q) | rot_bits(c, S, n + q); ge2 |= ones & mk; ones |= mk; }
        const uint32_t alive0 = p.alive;
        uint32_t marked = 0;                        // node positions to remove
        for (int pos = 0; pos < m; ++pos) {
            const uint32_t r = ord_get(p, pos);
            if ((ge2 >> r) & 1u) continue;          // weight >= 2: not trivial (pauli_network.rs:83-97)
            const uint32_t anti = (X[PX_ANTI + (r >> 1)] >> ((r & 1) * 16)) & 0xFFFFu;   // earlier rotations that anticommute
            if ((anti & alive0) != 0) continue;     // has an outgoing edge: not in the front layer (pauli_dag.rs:47-57)
            marked |= 1u << pos;
            p.alive &= ~(1u << r);                  // set_column(zeros) (pauli_network.rs:153-156)
            if (!((ones >> r) & 1u)) { err |= QG_FLAG_BAD_ROTATION; continue; }   // which_qubit().unwrap() panic in the reference
            int q = 0; uint32_t x = 0, z = 0;
            for (; q < n; ++q) { x = (rot_bits(c, S, q) >> r) & 1u; z = (rot_bits(c, S, n + q) >> r) & 1u; if (x | z) break; }
            const uint32_t axis = x ? (z ? 1u : 0u) : 2u;   // which_axis (121-137)
            hv[nh++] = (axis << 21) | ((uint32_t)q << 11) | (r << 1);
        }
        if (!marked) return;
        for (int pos = m - 1; pos >= 0; --pos)      // retain_nodes: high -> low, swap-remove
            if ((marked >> pos) & 1u) { ord_set(p, pos, ord_get(p, m - 1)); --m; }
        p.misc = (p.misc & 0x00FFFFFFu) | ((uint32_t)m << 24);
    }
}
// pauli_network.rs:196-207
template <class Wd>
__device__ __forceinline__ void pn_cnot(const DevCfg& c, const Wd& S, const Wd& X, PauliRegs& p, int i, int j, const Wd& hv, int& nh, uint32_t& err) {
    pn_row_xor(c, S, i, j);
    pn_row_xor(c, S, c.n + j, c.n + i);
    pn_clean(c, S, X, p, hv, nh, err);
}
// pauli_network.rs:225-260 as a fixed schedule  [one-qubit op] [up to three CNOTs] [one-qubit op]  instead of a switch over the
// eight gate kinds: the lanes of a warp hold different gates, and this way the warp runs the one-qubit routine at most twice
// and the CNOT + clean routine at most three times per step, whatever mix of gates its 32 environments drew.
//   H/S/Sdg/SX/SXdg(q0): pre            CX(q0,q1): cnot(q0,q1)
//   CZ(q0,q1) = h(q1), cnot(q0,q1), h(q1) (243-249)        SWAP(q0,q1) = cnot(q0,q1), cnot(q1,q0), cnot(q0,q1) (250-257)
template <class Wd>
__device__ void pn_act(const DevCfg& c, const Wd& S, const Wd& X, PauliRegs& p, int kind, int q0, int q1, const Wd& hv, int& nh, uint32_t& err) {
    const int pre = kind <= QG_SXDG ? pn_type_1q(kind) : (kind == QG_CZ ? 1 : 0);
    const int pre_q = kind == QG_CZ ? q1 : q0;
    const int ncnot = kind == QG_SWAP ? 3 : (kind == QG_CX || kind == QG_CZ ? 1 : 0);
    if (pre) pn_1q(c, S, p, pre, pre_q);
    for (int k = 0; k < ncnot; ++k) {
        const bool flip = k == 1;
        pn_cnot(c, S, X, p, flip ? q1 : q0, flip ? q0 : q1, hv, nh, err);
    }
    if (kind == QG_CZ) pn_1q(c, S, p, 1, q1);
}
// pauli_network.rs:167-173
template <class Wd>
__device__ __forceinline__ bool pn_solved(const DevCfg& c, const Wd& S, const PauliRegs& p) {
    if ((p.misc >> 24) != 0) return false;
    const int D = 2 * c.n, RW = c.CW >> 5;
    uint32_t diff = 0;
    for (int r = 0; r < D; ++r) {
        const uint32_t lo = S[r * RW];
        if (D <= 32) diff |= (D == 32 ? lo : (lo & ((1u << D) - 1u))) ^ (1u << r);
        else {
            const uint32_t hi = S[r * RW + 1] & ((1u << (D - 32)) - 1u);      // D <= 62 (2n + rotations <= 64)
            diff |= (lo ^ (r < 32 ? (1u << r) : 0u)) | (hi ^ (r >= 32 ? (1u << (r - 32)) : 0u));
        }
    }
    return diff == 0;
}
// observe(): pad_and_collect (pauli.rs:411-437) + apply_perm_to_obs (445-485) -> obs bit stream O, rows of obs_cols =
// 2n + max_rotations bits written one after the other through a 64-bit accumulator.
template <class Wd>
__device__ void pn_build_obs(const DevCfg& c, const Wd& S, const PauliRegs& p, const Wd& O, int perm_idx) {
    const int n = c.n, D = 2 * n, RW = c.CW >> 5;
    const int m = min((int)(p.misc >> 24), c.max_rot);
    const uint8_t* perm = (c.nperms > 0) ? (c.qperms + (size_t)perm_idx * n) : nullptr;
    if (!perm && c.obs_cols <= 32 && c.max_rot <= 8) {
        // the usual shape (C4: 20 + 5 columns): one observation row fits a word.  The DAG-order gather of the rotation bits runs over
        // eight shift amounts computed once per step (positions >= m read bit 31 of a < 2^16 value: zero) and a row is ONE append
        // (2 500 -> ~900 instructions per env-step, ncu source counters in profiles/r2_*)
        uint32_t sh[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) sh[i] = (i < m) ? ((p.ord0 >> (4 * i)) & 15u) : 31u;
        const uint32_t tmask = (1u << D) - 1u;                      // D <= 31 here
        unsigned long long acc = 0; int fill = 0, ow = 0;
        for (int r = 0; r < D; ++r) {
            const uint32_t t = S[r * RW] & tmask, rb = rot_bits(c, S, r);
            uint32_t rot = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) rot |= ((rb >> sh[i]) & 1u) << i;
            acc |= (unsigned long long)(t | (rot << D)) << fill; fill += c.obs_cols;
            if (fill >= 32) { O[ow++] = (uint32_t)acc; acc >>= 32; fill -= 32; }
        }
        if (fill > 0) O[ow++] = (uint32_t)acc;
        for (; ow < c.OW; ++ow) O[ow] = 0;
        return;
    }
    unsigned long long acc = 0; int fill = 0, ow = 0;
    auto append = [&](uint32_t v, int len) {       // len in 1..32, v has no bits above len
        acc |= (unsigned long long)v << fill; fill += len;
        if (fill >= 32) { O[ow++] = (uint32_t)acc; acc >>= 32; fill -= 32; }
    };
    for (int r = 0; r < D; ++r) {
        int src = r;
        if (perm) src = (r < n) ? (int)perm[r] : n + (int)perm[r - n];
        const uint32_t lo = S[src * RW], hi = D > 32 ? S[src * RW + 1] : 0u;
        uint32_t l0 = lo, l1 = hi;
        if (perm) {                                  // tableau columns move with the qubits too (pauli.rs:470-480)
            const unsigned long long bits = ((unsigned long long)hi << 32) | lo;
            unsigned long long o = 0;
            for (int col = 0; col < D; ++col) {
                const int sc = (col < n) ? (int)perm[col] : n + (int)perm[col - n];
                o |= ((bits >> sc) & 1ull) << col;
            }
            l0 = (uint32_t)o; l1 = (uint32_t)(o >> 32);
        }
        if (D <= 32) append(D == 32 ? l0 : (l0 & ((1u << D) - 1u)), D);
        else { append(l0, 32); append(l1 & ((1u << (D - 32)) - 1u), D - 32); }
        const uint32_t rb = rot_bits(c, S, src);
        uint32_t rot = 0, ow0 = p.ord0;
        for (int i = 0; i < m; ++i) {                // active rotations in DAG node order (pauli.rs:411-437)
            if (i == 8) ow0 = p.ord1;
            rot |= ((rb >> (ow0 & 15u)) & 1u) << i;
            ow0 >>= 4;
        }
        append(rot, c.max_rot);
    }
    if (fill > 0) O[ow++] = (uint32_t)acc;
    for (; ow < c.OW; ++ow) O[ow] = 0;
}

// ---- the fused kernel ----------------------------------------------------------------------------------
// Work decomposition: one WARP owns a tile of 32 consecutive environments (lane == environment in phase 1) and a
// private shared-memory region [word][kStride]; there is no block-level barrier, so warps drift apart and the
// latency-bound phase 1 of one warp overlaps the store-bound phase 2 of the others on the same SM.
// The records are loaded once, then `nsteps` steps are played from a resident action stream (nsteps == 1 is the
// policy-in-the-loop step; nsteps == T replays a whole episode without the state leaving the SM), then written back.
constexpr int kStride = 33;          // odd word stride: bank = (word + lane) % 32 -> conflict free both for per-lane private
                                     // access with a warp-uniform word and for the expander's broadcast reads of one env
constexpr int kWarpsPerCta = 2;

__device__ __forceinline__ void cp_async_4(uint32_t* smem_dst, const uint32_t* gsrc) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
// programmatic dependent launch: let the next grid of the stream start its prologue, and wait for the previous one
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

// store flavour of the observation / mask slabs (compile-time switch for A/B runs): 0 = st.global.cs (streaming, evict first),
// 1 = plain st.global, 2 = st.global.wt, 3 / 4 = L2 cache hint evict_last / evict_unchanged
// Measured (replay, 65 536 envs, profiles/r1_v22_store_policy.txt): plain stores are 2.4 % faster than .cs on C3 (also at 1 M envs),
// 0.7-0.9 % slower on C1 / C5 and 2 % slower for single-step launches; evict_unchanged equals plain, evict_last is 4 % slower.  So
// QG_STORE == 1 uses plain stores only in the whole-row fast path of replay launches (st_rows) and .cs everywhere else.  A
// persisting-L2 window over the action stream is much worse (40 MB set aside: -20 %): the write stream lives off the L2 capacity it
// can buffer in.
#ifndef QG_STORE
#define QG_STORE 1
#endif
#if QG_STORE == 3 || QG_STORE == 4
__device__ __forceinline__ unsigned long long l2_policy() {
    unsigned long long pol;
#if QG_STORE == 3
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#else
    asm("createpolicy.fractional.L2::evict_unchanged.b64 %0, 1.0;" : "=l"(pol));
#endif
    return pol;
}
__device__ __forceinline__ void st_hint(float4* p, const float4& v) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(l2_policy()) : "memory");
}
__device__ __forceinline__ void st_hint(uint4* p, const uint4& v) {
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(l2_policy()) : "memory");
}
#endif
// the action / coin streams are read once; evict-first loads (QG_LDCS) were measured: no change (1.620 vs 1.621 ms)
#ifdef QG_LDCS
#define QG_LD_STREAM(p) __ldcs(p)
#else
#define QG_LD_STREAM(p) (*(p))
#endif
template <class V>
__device__ __forceinline__ void st_slab(V* p, const V& v) {
#if QG_STORE == 0 || QG_STORE == 1
    __stcs(p, v);
#elif QG_STORE == 2
    __stwt(p, v);
#else
    st_hint(p, v);
#endif
}
// the whole-row fast path of a replay launch (see QG_STORE above): plain stores
template <bool PLAIN, class V>
__device__ __forceinline__ void st_rows(V* p, const V& v) {
#if QG_STORE == 1
    if (PLAIN) *p = v; else __stcs(p, v);
#else
    st_slab(p, v);
#endif
}
__device__ __forceinline__ float4 nibble_to_float4(uint32_t nib) {
    float4 f;
    f.x = (nib & 1u) ? 1.0f : 0.0f; f.y = (nib & 2u) ? 1.0f : 0.0f; f.z = (nib & 4u) ? 1.0f : 0.0f; f.w = (nib & 8u) ? 1.0f : 0.0f;
    return f;
}
// nibble -> float4 table in shared memory: entry (nib, copy) at float4 index nib * 8 + copy, copy = lane & 7.  A quarter
// warp (8 consecutive lanes, the unit a 128-bit shared load is served in) then touches 8 different 16-byte bank groups
// whatever the nibbles are: conflict free.  Every warp writes the whole table itself before it reads it (the warps of a CTA
// write identical values), so no block barrier is needed.
constexpr int kLutWords = 16 * 8 * 4;
__device__ __forceinline__ void lut_fill(uint32_t* lut, int lane) {
#pragma unroll
    for (int i = lane; i < 128; i += 32) reinterpret_cast<float4*>(lut)[i] = nibble_to_float4((uint32_t)i >> 3);
    __syncwarp();
}
__device__ __forceinline__ float4 lut_get(const uint32_t* lut_lane /* lut + (lane & 7) * 4 */, uint32_t nib) {
    return *reinterpret_cast<const float4*>(lut_lane + (nib << 5));
}
// 4 bits at bit offset `off` of environment e's observation bit stream (words at bits[w * kStride + e])
template <int kStride>
__device__ __forceinline__ uint32_t stream_nibble(const uint32_t* bits, uint32_t e, uint32_t off) {
    const uint32_t w = off >> 5, s = off & 31u;
    const uint32_t lo = bits[w * kStride + e];
    const uint32_t hi = (s > 28u) ? bits[(w + 1) * kStride + e] : 0u;
    return __funnelshift_r(lo, hi, s);
}

// ---- the tile's observations as ONE bit stream ------------------------------------------------------------------------------------
// The warp's slab of the [B][obs] float tensor is contiguous, so bit (e * obs + i) of the concatenation of its environments' observation
// bits is float number (e * obs + i) of the slab, whatever obs is.  With the concatenated stream in shared memory (cnt * obs / 32 words)
// the expansion is the same loop for every observation size: lane l always holds nibble (l & 7) of words (l >> 3) + 4k — one LDS
// (broadcast within a quarter warp), a shift, one table load and one 16-byte store per 512 bytes — instead of the per-float4
// (environment, offset) bookkeeping that observations which are not whole words per environment used to need (C1: 81, C4: 500, C5: 729
// entries: 40 instructions per store before, 5 after; ncu instruction counts in profiles/r2_*).
// cat_gather builds the stream from the per-environment streams bits[word * kStride + env] (any obs; used by PauliNetwork); Permutation sets
// its n one-hot bits per environment straight into the concatenated stream (cat_onehot), skipping the per-environment stream altogether.
template <int kStride>
__device__ __forceinline__ void cat_gather(const uint32_t* bits, uint32_t* cat, uint32_t cnt, uint32_t obs, uint64_t magic_obs, int lane) {
    const uint32_t total = cnt * obs, nwords = (total + 31u) >> 5;
    for (uint32_t W = lane; W < nwords; W += 32) {
        uint32_t e = fastdiv40(W << 5, magic_obs), off = (W << 5) - e * obs, v = 0, filled = 0;
        while (filled < 32u && e < cnt) {
            const uint32_t len = min(32u - filled, obs - off), w = off >> 5, sft = off & 31u;
            const uint32_t lo = bits[w * kStride + e], hi = (sft + len > 32u) ? bits[(w + 1) * kStride + e] : 0u;
            uint32_t x = __funnelshift_r(lo, hi, sft);
            if (len < 32u) x &= (1u << len) - 1u;
            v |= x << filled;
            filled += len; off += len;
            if (off == obs) { off = 0; ++e; }
        }
        cat[W] = v;
    }
    __syncwarp();
}
template <class Wd>
__device__ __forceinline__ void cat_onehot(const DevCfg& c, const Wd& S, uint32_t* cat, uint32_t cnt, bool live, int lane) {
    const uint32_t obs = (uint32_t)c.obs_size, nwords = (cnt * obs + 31u) >> 5;
    for (uint32_t W = lane; W < nwords; W += 32) cat[W] = 0;
    __syncwarp();
    if (live) {
        uint32_t bit = (uint32_t)lane * obs;                      // row i of env `lane` starts at bit lane * obs + i * n (permutation.rs:241-243)
        for (int i = 0; i < c.n; ++i, bit += (uint32_t)c.n) { const uint32_t b = bit + get8(S, i); atomicOr(cat + (b >> 5), 1u << (b & 31u)); }
    }
    __syncwarp();
}
template <bool PLAIN>
__device__ __forceinline__ void expand_cat(const uint32_t* cat, const uint32_t* lut, float* out, uint32_t total /* cnt * obs floats */, int lane) {
    const bool vec_ok = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
    const uint32_t nvec = vec_ok ? (total >> 2) : 0u, sh = ((uint32_t)lane & 7u) << 2;
    const uint32_t* const lut_lane = lut + ((lane & 7) << 2);
    const uint32_t* src = cat + ((uint32_t)lane >> 3);
    float4* o = reinterpret_cast<float4*>(out) + lane;
#pragma unroll 4
    for (uint32_t j = lane; j < nvec; j += 32, src += 4, o += 32) st_rows<PLAIN>(o, lut_get(lut_lane, (*src >> sh) & 15u));
    for (uint32_t f = (nvec << 2) + lane; f < total; f += 32) out[f] = ((cat[f >> 5] >> (f & 31u)) & 1u) ? 1.0f : 0.0f;
}

// Phase 2a: bits -> floats.  The warp's slab out[0 .. cnt*obs_size) is contiguous in the [B][obs_size] tensor; lane l
// stores the float4 number l, l+32, ... (512 contiguous bytes per warp instruction).  (e, v) = (environment, float4 within
// the environment) of a lane's float4 is tracked incrementally: advancing 32 float4s adds (q, r) with one conditional wrap,
// so the loop has no division; the four floats come from the shared-memory table with one 128-bit load.
template <int MODE, int kStride>
__device__ __forceinline__ void expand_obs(const uint32_t* bits, const uint32_t* lut, float* out, uint32_t cnt, uint32_t obs, uint32_t en_bits, int lane,
                                           uint32_t magic_obs4 /*ceil(2^32/(obs/4)) or 0*/, uint64_t magic_obs, uint32_t q4, uint32_t r4, bool plain_rows) {
    // 16-byte stores need an aligned slab: always true for the engine's own [B][obs] tensors; a ring slot of an odd-sized
    // batch may start off the grid, then everything goes through the scalar tail loop
    const bool vec_ok = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
    const uint32_t* const lut_lane = lut + ((lane & 7) << 2);
    float4* const out4 = reinterpret_cast<float4*>(out);
    if (vec_ok && (obs & 127u) == 0) {
        // whole 512-byte warp stores per environment: lane l always holds nibble (l & 7) of words (l >> 3) + 4k of the current
        // environment, so the loop is one LDS (broadcast within a quarter warp) + shift + table load + store per 512 bytes
        const uint32_t K = obs >> 7, VPE = obs >> 2, sh = ((uint32_t)lane & 7u) << 2;
        const uint32_t* src = bits + ((uint32_t)lane >> 3) * kStride;
        float4* o = out4 + lane;
        // measured dead ends at 65 536 envs (profiles/r1_v15_ablation*.jsonl, r1_v16_ablation_pipe.jsonl): floats from selects
        // instead of the table (no change), the words of 8 environments read ahead of 16 back-to-back stores (1.7 % slower),
        // the L1 / shared-memory carve-out (no change), more storing warps per tile (tools/store_pattern_probe.cu: no change)
        auto rows = [&](auto plain) {
            constexpr bool PLAIN = decltype(plain)::value;
            if (K == 2) {
#pragma unroll 4
                for (uint32_t e = 0; e < cnt; ++e, o += 64) {
                    if (MODE == MODE_SEARCH && !((en_bits >> e) & 1u)) continue;
                    const uint32_t w0 = src[e], w1 = src[4 * kStride + e];
                    st_rows<PLAIN>(o, lut_get(lut_lane, (w0 >> sh) & 15u));
                    st_rows<PLAIN>(o + 32, lut_get(lut_lane, (w1 >> sh) & 15u));
                }
            } else {
                for (uint32_t e = 0; e < cnt; ++e, o += VPE) {
                    if (MODE == MODE_SEARCH && !((en_bits >> e) & 1u)) continue;
#pragma unroll 4
                    for (uint32_t k = 0; k < K; ++k) st_rows<PLAIN>(o + (k << 5), lut_get(lut_lane, (src[(k << 2) * kStride + e] >> sh) & 15u));
                }
            }
        };
        if (plain_rows) rows(std::true_type{}); else rows(std::false_type{});
    } else if (vec_ok && (obs & 31u) == 0) {
        // whole words per environment: a lane's nibble position inside its word never changes (r4 is a multiple of 8)
        const uint32_t VPE = obs >> 2, total = cnt * VPE, sh = ((uint32_t)lane & 7u) << 2;
        uint32_t e = (VPE == 1) ? (uint32_t)lane : __umulhi((uint32_t)lane, magic_obs4), v = (uint32_t)lane - e * VPE;
        const uint32_t* src = bits + (v >> 3) * kStride + e;
        const int32_t dstep = (int32_t)(q4 + (r4 >> 3) * kStride), dwrap = 1 - (int32_t)(VPE >> 3) * kStride;
        if (r4 == 0) {          // VPE divides 32: the lane keeps its word column and only walks the environments
#pragma unroll 4
            for (uint32_t j = lane; j < total; j += 32) {
                if (MODE != MODE_SEARCH || ((en_bits >> e) & 1u)) st_slab(out4 + j, lut_get(lut_lane, (*src >> sh) & 15u));
                src += dstep; e += q4;
            }
        } else {
#pragma unroll 4
            for (uint32_t j = lane; j < total; j += 32) {
                if (MODE != MODE_SEARCH || ((en_bits >> e) & 1u)) st_slab(out4 + j, lut_get(lut_lane, (*src >> sh) & 15u));
                src += dstep; e += q4; v += r4;
                if (v >= VPE) { v -= VPE; src += dwrap; ++e; }
            }
        }
    } else if (vec_ok && (obs & 3u) == 0) {
        // a float4 never straddles two environments
        const uint32_t VPE = obs >> 2, total = cnt * VPE;
        uint32_t e = (VPE == 1) ? (uint32_t)lane : __umulhi((uint32_t)lane, magic_obs4), v = (uint32_t)lane - e * VPE;
#pragma unroll 4
        for (uint32_t j = lane; j < total; j += 32) {
            if (MODE != MODE_SEARCH || ((en_bits >> e) & 1u)) {
                const uint32_t nib = bits[(v >> 3) * kStride + e] >> ((v & 7u) << 2);
                st_slab(out4 + j, lut_get(lut_lane, nib & 15u));
            }
            e += q4; v += r4;
            if (v >= VPE) { v -= VPE; ++e; }
        }
    } else {
        const uint32_t total = cnt * obs, nvec = (vec_ok && obs >= 4u) ? (total >> 2) : 0u;
        uint32_t e = fastdiv40((uint32_t)lane << 2, magic_obs), off = ((uint32_t)lane << 2) - e * obs;
        const uint32_t q = 128u / obs, r = 128u - q * obs;
        if (nvec) {
#pragma unroll 2
            for (uint32_t j = lane; j < nvec; j += 32) {
                uint32_t nib = stream_nibble<kStride>(bits, e, off);
                const bool straddle = off + 4u > obs;                 // the float4 ends in environment e+1
                if (straddle) { const uint32_t k = obs - off; nib = (nib & ((1u << k) - 1u)) | (bits[e + 1] << k); }
                const bool on = (MODE != MODE_SEARCH) || (((en_bits >> e) & 1u) && (!straddle || ((en_bits >> (e + 1)) & 1u)));
                if (on) st_slab(out4 + j, lut_get(lut_lane, nib & 15u));
                else {
                    uint32_t ee = e, oo = off;
                    for (int k = 0; k < 4; ++k) { if ((en_bits >> ee) & 1u) out[(j << 2) + k] = ((nib >> k) & 1u) ? 1.0f : 0.0f; if (++oo == obs) { oo = 0; ++ee; } }
                }
                e += q; off += r;
                if (off >= obs) { off -= obs; ++e; }
            }
        }
        // elements not covered by whole float4s (ragged last tile, or obs < 4)
        for (uint32_t f = (nvec << 2) + lane; f < total; f += 32) {
            const uint32_t ee = fastdiv40(f, magic_obs), oo = f - ee * obs;
            if (MODE != MODE_SEARCH || ((en_bits >> ee) & 1u)) out[f] = ((bits[(oo >> 5) * kStride + ee] >> (oo & 31u)) & 1u) ? 1.0f : 0.0f;
        }
    }
}

// Phase 2b: masks() = [!success; A] per environment (clifford.rs:349-351) as a uint8 [B][A] slab, 16-byte stores.
// G = bytes per granule that cannot straddle two environments (4 when A % 4 == 0, else 1).
template <int MODE, int G>
__device__ __forceinline__ void expand_mask(uint8_t* out, uint32_t cnt, uint32_t A, uint32_t mask_bits, uint32_t en_bits, int lane, uint64_t magic_A) {
    const uint32_t total = cnt * A, nvec = (reinterpret_cast<uintptr_t>(out) & 15u) ? 0u : (total >> 4);   // whole 16-byte vectors of the (aligned) slab
    if (MODE != MODE_SEARCH) {
        // the usual case: the 32 environments agree (nobody solved yet, or all solved) -> a plain fill of the slab
        const uint32_t live = cnt >= 32u ? 0xFFFFFFFFu : ((1u << cnt) - 1u);
        if (mask_bits == live || mask_bits == 0u) {
            const uint32_t w = mask_bits ? 0x01010101u : 0u;
            const uint4 w4 = make_uint4(w, w, w, w);
            for (uint32_t j = lane; j < nvec; j += 32) st_slab(reinterpret_cast<uint4*>(out) + j, w4);
            for (uint32_t b = (nvec << 4) + lane; b < total; b += 32) out[b] = (uint8_t)(w & 1u);
            return;
        }
    }
    const uint32_t P = A / G;                                     // granules per environment
    const uint32_t g0 = ((uint32_t)lane << 4) / G;                // first granule of this lane's first vector
    uint32_t e = fastdiv40(g0 * G, magic_A), off = g0 - e * P;
    const uint32_t step = 512u / G, q = step / P, r = step - q * P;
    for (uint32_t j = lane; j < nvec; j += 32) {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        uint32_t ee = e, oo = off; bool all_on = true;
#pragma unroll
        for (int k = 0; k < 16 / G; ++k) {
            const uint32_t bit = (mask_bits >> ee) & 1u;
            if (MODE == MODE_SEARCH && !((en_bits >> ee) & 1u)) all_on = false;
            if (G == 4) w[k] = bit ? 0x01010101u : 0u; else w[k >> 2] |= bit << ((k & 3) * 8);
            if (++oo == P) { oo = 0; ++ee; }
        }
        if (MODE != MODE_SEARCH || all_on) st_slab(reinterpret_cast<uint4*>(out) + j, make_uint4(w[0], w[1], w[2], w[3]));
        else {
            uint32_t e2 = e, o2 = off;
            for (int k = 0; k < 16 / G; ++k) {
                if ((en_bits >> e2) & 1u) { for (int b = 0; b < G; ++b) out[(j << 4) + k * G + b] = (uint8_t)((mask_bits >> e2) & 1u); }
                if (++o2 == P) { o2 = 0; ++e2; }
            }
        }
        e += q; off += r;
        if (off >= P) { off -= P; ++e; }
    }
    for (uint32_t b = (nvec << 4) + lane; b < total; b += 32) {   // ragged last tile
        const uint32_t ee = fastdiv40(b, magic_A);
        if (MODE != MODE_SEARCH || ((en_bits >> ee) & 1u)) out[b] = (uint8_t)((mask_bits >> ee) & 1u);
    }
}

// hand-over barriers of a warp pair: hardware named barriers 0..3 of the CTA (full[0..1] = 0, 1; empty[0..1] = 2, 3; 64 threads each: the 32
// lanes of the warp that is done arrive, the 32 of the waiting warp sync and sleep in hardware until then).  Shared-memory mbarriers with a
// try_wait / nanosleep loop measure the same within 0.5 % (profiles/r2_v26_pair_ab.txt) and are kept as a tools build.
#ifdef QG_PAIR_MBARRIER      // (tools A/B build)
__device__ __forceinline__ void pair_arrive(uint64_t* bars, int idx, int lane) {
    __syncwarp();
    // idx >= 2: the store warp frees a buffer it has only READ (its loads have returned: their values fed the stores) — a relaxed arrive
    if (lane == 0) {
        if (idx >= 2) asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];\n" ::"r"((uint32_t)__cvta_generic_to_shared(bars + idx)) : "memory");
        else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"((uint32_t)__cvta_generic_to_shared(bars + idx)) : "memory");
    }
}
__device__ __forceinline__ void pair_wait(uint64_t* bars, int idx, uint32_t parity) {
    const uint32_t addr = (uint32_t)__cvta_generic_to_shared(bars + idx);
    uint32_t ok = 0;
    while (true) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (ok) break;
        __nanosleep(128);
    }
}
#else
// (immediate barrier numbers 0..3: with the number in a register ptxas reserves all 16 barriers for the CTA and the SM holds 4 CTAs instead of 16)
__device__ __forceinline__ void pair_arrive(uint64_t*, int idx, int) {
    switch (idx) {
        case 0: asm volatile("bar.arrive 0, 64;\n" ::: "memory"); break;
        case 1: asm volatile("bar.arrive 1, 64;\n" ::: "memory"); break;
        case 2: asm volatile("bar.arrive 2, 64;\n" ::: "memory"); break;
        default: asm volatile("bar.arrive 3, 64;\n" ::: "memory"); break;
    }
}
__device__ __forceinline__ void pair_wait(uint64_t*, int idx, uint32_t) {
    switch (idx) {
        case 0: asm volatile("bar.sync 0, 64;\n" ::: "memory"); break;
        case 1: asm volatile("bar.sync 1, 64;\n" ::: "memory"); break;
        case 2: asm volatile("bar.sync 2, 64;\n" ::: "memory"); break;
        default: asm volatile("bar.sync 3, 64;\n" ::: "memory"); break;
    }
}
#endif

// Rows of the action / coin streams that the copy engine is still bringing from the host (qg_replay_host_packed): the warp that is about to read
// row `step` waits until the chunk that starts there has landed (the flag is a 4-byte copy queued behind the chunk's copies on the same stream).
__device__ __forceinline__ void wait_input_chunk(const StepArgs& a, int step, int lane) {
    int k = -1;
#pragma unroll
    for (int i = 0; i < 4; ++i) if (step == a.in_chunk[i]) k = i;
    if (k < 0) return;
    if (lane == 0) {
        long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(a.in_flags + k) : "memory");
            if (v) break;
            __nanosleep(256);
            long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 10000000000ll) break;          // 10 s: a copy that never comes must not hang the device
        }
    }
    __syncwarp();
}

// The work of ONE warp on its tile of `cnt` (<= 32) consecutive environments starting at e0: record load, `a.nsteps` steps
// (phase 1 + phase 2 each), record write-back.  wbase: the warp's private shared-memory region (a.sm_warp_words words), lut: the
// CTA's nibble -> float4 table (only read when a.obs is set).  Returns the ballot of the environments that were stepped in the
// last step (MODE_SEARCH: rollouts that were not final).  k_step calls it once per warp; the fused search kernel
// (qg_search_fused.cuh) calls it once per decision for the rollouts its CTA owns.
// resident: the warp's shared-memory region still holds the tile's records from its previous call (the fused search kernel calls
// it once per decision for the same environments): skip the load.  weights_tile: MODE_SEARCH action weights of the tile's
// environments, [cnt][A] starting at environment e0 (may point to shared memory), or null to read a.weights[env * A].
// fused (the one-launch search, which keeps calling for the same tile): the observation bit stream is built in shared memory even though
// no output tensor is given, the records are not written back to global memory (tile_writeback does that once, at the end), the running
// return is kept in ret_local[lane] (shared memory) instead of c.ret, and a resident Permutation's one-hot stream is patched (4 bits per
// SWAP) instead of rebuilt.
// EPW: environments per warp tile (32, or 16: twice the warps for the same batch, lanes 16..31 idle in phase 1 and at work in phase 2 —
// at 65 536 environments that is 28 instead of 14 warps per SM to overlap one warp's latency-bound step logic with the others' stores).
// The tile's shared-memory words are laid out [word][EPW + 1].
// TWIST: the launch may carry a twisted collector's action tables (a.act_perm); the fused search never does and compiles without that path.
template <int KIND, int MODE, int INV, int EPW = 32, int ROLE = 0, bool TWIST = true>
__device__ __forceinline__ uint32_t step_tile(const DevCfg& c, const StepArgs& a, uint32_t* const wbase, const uint32_t* const lut, const int lane,
                                              const int64_t e0, const int cnt, const bool resident = false, const float* const weights_tile = nullptr,
                                              const bool fused = false, float* const ret_local = nullptr) {
    constexpr int role = ROLE;             // compile-time: the solo kernels carry none of the pair code (their single-step launches are
                                           // latency-bound and lost 10-40 % to the larger code when the role was a run-time argument)
    // role (replay launches with a.pair): 0 = the warp does everything; 1 = step warp: plays the steps and hands every step's observation
    // bits + mask ballot to its partner through two buffers; 2 = store warp: expands them into the float / mask slabs.  The latency-bound
    // step logic of step t+1 then overlaps the stores of step t on the SAME tile without more environments per SM (full[b] / empty[b] named
    // barriers per buffer b = t & 1).
    constexpr int kStride = EPW + 1;       // (shadows the namespace constant: everything below indexes the tile with this launch's stride)
    typedef SmWords<kStride> Wd;
    const int64_t env = e0 + lane;
    const bool live = lane < cnt;
    const Wd R{wbase + lane};
    const Wd LG = R.at(c.off_lastg), LC = R.at(c.off_lastcx), S = R.at(c.off_state), X = R.at(c.off_extra);
    const Wd SCR{wbase + a.sm_scr + lane}, O{wbase + a.sm_obs + lane};
    const bool obs_from_O = (KIND == QG_ENV_PAULI_NETWORK) || (KIND == QG_ENV_PERMUTATION && c.OW > 0);
    const uint32_t* const obs_bits = wbase + (obs_from_O ? a.sm_obs : c.off_state * kStride);
    // dense observations that are not whole words per environment go through the tile's concatenated bit stream (expand_cat); search /
    // slot launches, whose tiles may skip environments, keep the per-element path
    const bool use_cat = MODE != MODE_SEARCH && a.obs && a.sm_cat >= 0 && !a.skip_negative && !fused;
    uint32_t* const cat = wbase + (a.sm_cat >= 0 ? a.sm_cat : 0);
    uint32_t* const pair_base = wbase + (role ? a.sm_pair : 0);
    uint32_t* const pair_hdr = pair_base + 2 * a.pair_words;                     // [2] mask ballots, then (8-byte aligned) the four mbarriers
    uint64_t* const pair_bar = reinterpret_cast<uint64_t*>(wbase + (role ? a.sm_pair_bar : 0));      // full[0], full[1], empty[0], empty[1]
    if constexpr (role == 2) {
        // ===== store warp of a pair =====
        const uint32_t en_all = cnt >= 32 ? 0xFFFFFFFFu : ((1u << cnt) - 1u);
        int slot2 = a.slot0;
        for (int t = 0; t < a.nsteps; ++t) {
            const int b = t & 1;
            pair_wait(pair_bar, b, (uint32_t)(t >> 1) & 1u);            // the step warp has filled buffer b
            const uint32_t* src = pair_base + b * a.pair_words;
            const uint32_t mask_bits2 = pair_hdr[b];
            float* out = a.obs + ((size_t)slot2 * c.B + (size_t)e0) * c.obs_size;
            if (use_cat) {
                if (KIND != QG_ENV_PERMUTATION) { cat_gather<kStride>(src, cat, (uint32_t)cnt, (uint32_t)c.obs_size, a.magic_obs, lane); src = cat; }
                expand_cat<true>(src, lut, out, (uint32_t)cnt * (uint32_t)c.obs_size, lane);
            } else {
                expand_obs<MODE, kStride>(src, lut, out, (uint32_t)cnt, (uint32_t)c.obs_size, en_all, lane, a.magic_vpe, a.magic_obs, a.exp_q, a.exp_r, true);
            }
            if (a.mask) {
                uint8_t* mout = a.mask + ((size_t)slot2 * c.B + (size_t)e0) * c.A;
                if ((c.A & 3) == 0) expand_mask<MODE, 4>(mout, (uint32_t)cnt, (uint32_t)c.A, mask_bits2, en_all, lane, a.magic_A);
                else expand_mask<MODE, 1>(mout, (uint32_t)cnt, (uint32_t)c.A, mask_bits2, en_all, lane, a.magic_A);
            }
            if (++slot2 == a.ring) slot2 = 0;
            pair_arrive(pair_bar, 2 + b, lane);                         // buffer b may be refilled
        }
        return en_all;
    }
    // MODE_SEARCH: the tile's action weights [cnt][A] are contiguous in global memory: the warp copies them into shared memory with coalesced
    // 4-byte cp.async (row stride A | 1: odd, so the lanes' rows start in different banks) instead of every lane walking its own row with a
    // 4*A-byte stride between lanes.  All of a lane's ~A copies are in flight at once, under the record load: through registers the loop held
    // four loads per lane in flight and a 65 536-env collector decision spent ~10 of its 21 us on their latency.
    const float* staged_wts = nullptr;
    if (MODE == MODE_SEARCH && !weights_tile && a.sm_wts >= 0) {
        float* w = reinterpret_cast<float*>(wbase + a.sm_wts);
        const uint32_t A = (uint32_t)c.A, rs = A | 1u, total = (uint32_t)cnt * A;
        const float* src = a.weights + (size_t)e0 * A;
        for (uint32_t i = lane; i < total; i += 32) {
            const uint32_t e = fastdiv40(i, a.magic_A);
            cp_async_4(reinterpret_cast<uint32_t*>(w + e * rs + (i - e * A)), reinterpret_cast<const uint32_t*>(src + i));
        }
        staged_wts = w;
    }
    uint32_t last_en_bits = 0;
    if (live && !resident) {
        const uint32_t* src = c.rec + (a.src_slot ? (int64_t)a.src_slot[env] : env);
#pragma unroll 4
        for (int w = 0; w < c.W; ++w, src += c.Bpad) cp_async_4(&R[w], src);       // all W loads in flight at once
        cp_async_wait_all();
    }
    if (MODE == MODE_SEARCH && staged_wts) { cp_async_wait_all(); __syncwarp(); }     // (lanes without an environment wait here; rows were written by all lanes)
    uint32_t depth = 0, flags = 0, tick = 0;
    PauliRegs pr{};
    if (live) {
        depth = R[HD_DEPTH]; flags = R[HD_FLAGS]; tick = R[HD_TICK];
        if (KIND == QG_ENV_PAULI_NETWORK) { pr.plo = X[PX_PLO]; pr.phi = X[PX_PHI]; pr.alive = X[PX_ALIVE]; pr.ord0 = X[PX_ORD0]; pr.ord1 = X[PX_ORD1]; pr.misc = X[PX_MISC]; }
    }
    bool dirty = false;                              // records changed: write them back at the end
    int slot = a.slot0;                              // observation / mask ring slot of this step

    // replay: the next step's action (and coin) is requested before this step's expansion, so its DRAM latency is hidden
    int next_action = -1; uint32_t next_coin = 0;
    // (rows still in flight from the host: L2-only loads — a line of L1 could hold the neighbouring row from before this one arrived)
    auto load_action = [&](size_t idx) {
        if (a.in_flags) return a.actions8 ? (int)__ldcg(a.actions8 + idx) : (int)__ldcg(a.actions + idx);
        return a.actions8 ? (int)QG_LD_STREAM(a.actions8 + idx) : (int)QG_LD_STREAM(a.actions + idx);
    };
    auto load_coin = [&](size_t idx) { return a.in_flags ? (uint32_t)__ldcg(a.coins + idx) : (uint32_t)QG_LD_STREAM(a.coins + idx); };
    if (MODE == MODE_STEP && a.in_flags) wait_input_chunk(a, 0, lane);
    if (MODE == MODE_STEP && live) {
        next_action = load_action((size_t)env);
        if (a.coins) next_coin = load_coin((size_t)env);
    }
    uint32_t acc_done = 0, acc_succ = 0;             // lane l: the tile's is_final / success ballots of step (t & ~31) + l (a.done_bits)
    for (int t = 0; t < a.nsteps; ++t) {
        uint32_t* const hand = pair_base + (t & 1) * a.pair_words;       // (role 1) this step's hand-over buffer
        if (role == 1 && t >= 2) pair_wait(pair_bar, 2 + (t & 1), (uint32_t)((t >> 1) - 1) & 1u);   // ... free again: the store warp is done with step t - 2
        const Wd Ob = (role == 1) ? Wd{hand + lane} : O;                 // where this step's per-env observation stream is built
        bool success = (flags & FL_SUCCESS) != 0, enabled = live;
        const uint32_t coin_in = next_coin;
        if (MODE == MODE_STEP && a.in_flags && t + 1 < a.nsteps) wait_input_chunk(a, t + 1, lane);       // (whole warp) row t + 1 is requested below
        if (live) {
            int action = -1;
            if (MODE == MODE_STEP) {
                action = next_action;
                if (a.skip_negative && action < 0) enabled = false;
                if (t + 1 < a.nsteps) {
                    next_action = load_action((size_t)(t + 1) * a.in_stride + env);
                    if (a.coins) next_coin = load_coin((size_t)(t + 1) * a.in_stride + env);
                }
            }
            if (MODE == MODE_SEARCH) {
                // twisterl-style rollout decision: skip rollouts that are final (is_final, clifford.rs:353)
                enabled = !(depth == 0 || success);
                // twisted collector: env action g's weight is wt[ap[g]] (the policy saw the twisted observation).  The arg-max and the sequential
                // inverse-CDF sum run over g in the same order as on the result of qg_twist_gather(weights, act_perm, twist): bit-identical picks
                const int32_t* const ap = (TWIST && a.act_perm && enabled) ? a.act_perm + (size_t)a.twist[env] * c.A : nullptr;
                if (enabled) {
                    const float* wt = weights_tile ? weights_tile + (size_t)lane * c.A
                                      : (staged_wts ? staged_wts + (size_t)lane * (c.A | 1) : a.weights + (size_t)env * c.A);
                    auto pick = [&](auto w_at) {
                        int act;
                        if (a.deterministic) {
                            float best = w_at(0); act = 0;
                            for (int k = 1; k < c.A; ++k) { const float v = w_at(k); if (v > best) { best = v; act = k; } }
                        } else {
                            float total = 0.0f;
#pragma unroll 4
                            for (int k = 0; k < c.A; ++k) total = __fadd_rn(total, w_at(k));
                            const uint32_t raw = philox_draw(seed_of(c), (uint64_t)(c.first_id + env), tick, STREAM_SAMPLE);
                            if (!(total > 0.0f)) act = (int)__umulhi(raw, (uint32_t)c.A);
                            else {
                                const float target = __fmul_rn((float)(raw >> 8) * (1.0f / 16777216.0f), total);
                                float cum = 0.0f; act = c.A - 1;
#pragma unroll 4
                                for (int k = 0; k < c.A; ++k) { cum = __fadd_rn(cum, w_at(k)); if (cum > target) { act = k; break; } }
                            }
                        }
                        return act;
                    };
                    if constexpr (TWIST) { if (ap) action = pick([&](int k) { return wt[__ldg(ap + k)]; }); else action = pick([&](int k) { return wt[k]; }); }
                    else action = pick([&](int k) { return wt[k]; });
                }
                if (a.chosen) a.chosen[env] = enabled ? action : -1;
                if constexpr (TWIST) { if (a.policy_chosen) a.policy_chosen[env] = enabled ? (ap ? __ldg(ap + action) : action) : -1; }
            }

            int oh_q0 = -1, oh_q1 = -1;                 // Permutation, fused + resident: the SWAP this step played (one-hot stream patch)
            bool oh_full = !(fused && resident);
            if (MODE != MODE_OBSERVE && enabled) {
                uint32_t err = 0;
                float penalty = 0.0f;
                int nh = 0;                                     // rotations harvested by this step (PauliNetwork)
                int act = action;
                if (act < 0) { err |= QG_FLAG_BAD_ACTION; act = 0x7FFFFFFF; }
                if (KIND == QG_ENV_PAULI_NETWORK && c.nperms > 0 && act < c.A)
                    act = (int)c.aperms[(size_t)(pr.misc & 0xFFFFu) * c.A + act];       // pauli.rs:594-599
                const bool valid = act < c.A;
                uint32_t sol_len = flags >> FL_LEN_SHIFT;
                auto push = [&](uint32_t v) {
                    if ((int)sol_len < c.sol_cap) { c.sol[(size_t)sol_len * c.Bpad + env] = v; ++sol_len; }
                    else err |= QG_FLAG_SOLUTION_OVERFLOW;
                };
                if (valid) {
                    const uint32_t g = __ldg(c.gates + act);
                    const int kind = (int)(g & 0xFFu), q0 = (int)((g >> 8) & 0xFFu), q1 = (int)((g >> 16) & 0xFFu);
                    Counts prev{R[HD_NCNOTS], R[HD_NGATES], R[HD_LAYERS] & 0xFFFFu, R[HD_LAYERS] >> 16};
                    Counts now = prev;
                    met_gate(LG, LC, c.n, kind, q0, q1, now, err);
                    penalty = weighted_delta(c, now, prev);
                    R[HD_NCNOTS] = now.nc; R[HD_NGATES] = now.ng; R[HD_LAYERS] = (now.nl & 0xFFFFu) | (now.nlc << 16);
                    if (KIND == QG_ENV_PAULI_NETWORK) pn_act(c, S, X, pr, kind, q0, q1, SCR, nh, err);
                    else apply_gate_state<KIND>(c, S, kind, q0, q1);
                    if (KIND == QG_ENV_PERMUTATION && kind == QG_SWAP) { oh_q0 = q0; oh_q1 = q1; }
                }
                // solution log: Permutation only for valid actions (permutation.rs:210-216), LF/Clifford always
                // (linear_function.rs:315-321, clifford.rs:334-340), PauliNetwork gate + harvested rotations (pauli.rs:612-627)
                if (c.track) {
                    if (KIND == QG_ENV_PAULI_NETWORK) {
                        if (valid) {
                            push((uint32_t)act);
                            if (nh > 0) {
                                uint32_t ylo = 0, yhi = 0;      // #Y per rotation mod 4 (pauli.rs:125-133), after the whole act()
                                for (int q = 0; q < c.n; ++q) { const uint32_t y = rot_bits(c, S, q) & rot_bits(c, S, c.n + q); const uint32_t cy = ylo & y; ylo ^= y; yhi ^= cy; }
                                for (int k = 0; k < nh; ++k) {
                                    const uint32_t h = SCR[k], r = (h >> 1) & 0xFu;
                                    const uint32_t bp = ((pr.plo >> r) & 1u) | (((pr.phi >> r) & 1u) << 1);
                                    const uint32_t ys = ((ylo >> r) & 1u) | (((yhi >> r) & 1u) << 1);
                                    const uint32_t ph = (bp - ys) & 3u;
                                    push(0x80000000u | h | (ph == 2u ? 0u : 1u));
                                }
                            }
                        }
                    } else if (KIND != QG_ENV_PERMUTATION || valid) {
                        push(((uint32_t)action & 0x7FFFFFFFu) | ((flags & FL_INVERTED) ? 0x80000000u : 0u));
                    }
                }
                depth = depth > 0 ? depth - 1 : 0;              // saturating_sub
                if (KIND != QG_ENV_PAULI_NETWORK && c.add_inverts) {
                    bool coin;
                    if (a.coins) coin = (MODE == MODE_STEP) ? (coin_in != 0) : (a.coins[(size_t)t * a.in_stride + env] != 0);
                    else coin = (philox_draw(seed_of(c), (uint64_t)(c.first_id + env), tick, STREAM_COIN) >> 31) != 0;
                    if (coin) {
                        if (KIND == QG_ENV_PERMUTATION) { invert_perm(c, S, SCR); flags ^= FL_INVERTED; oh_full = true; }
                        else {
                            bool inverted;
                            if constexpr (INV == 0) inverted = invert_matrix(c, S, SCR, SCR.at(c.SW));
                            else if (KIND == QG_ENV_CLIFFORD && a.symplectic) { symplectic_invert_rows<INV>(S, c.n); inverted = true; }
                            else inverted = gf2_invert_rows<INV>(S, c.D);
                            if (inverted) flags ^= FL_INVERTED; else err |= QG_FLAG_SINGULAR;
                        }
                    }
                }
                success = (KIND == QG_ENV_PAULI_NETWORK) ? pn_solved(c, S, pr) : solved_state<KIND>(c, S);
                float reward = __fsub_rn(success ? 1.0f : 0.0f, penalty);
                if (KIND == QG_ENV_PAULI_NETWORK) reward = __fadd_rn(reward, __fmul_rn(c.plr, (float)nh));   // pauli.rs:634
                flags = (flags & (FL_INVERTED | (0xFFu << FL_ERR_SHIFT))) | (success ? FL_SUCCESS : 0u) | (err << FL_ERR_SHIFT) | (sol_len << FL_LEN_SHIFT);
                tick += 1;
                R[HD_REWARD] = __float_as_uint(reward);
                dirty = true;
                if (MODE == MODE_SEARCH) {
                    if (ret_local) ret_local[lane] = __fadd_rn(ret_local[lane], reward);
                    else c.ret[env] = __fadd_rn(c.ret[env], reward);
                }
                if (a.reward) a.reward[(size_t)t * a.out_stride + env] = reward;
            }
            if (MODE == MODE_OBSERVE && a.reward) a.reward[env] = __uint_as_float(R[HD_REWARD]);
            if (enabled) {
                if (a.done) a.done[(size_t)t * a.out_stride + env] = (depth == 0 || success) ? 1 : 0;
                if (a.success) a.success[(size_t)t * a.out_stride + env] = success ? 1 : 0;
            }

            // observe(): build the observation bit stream where it is not the state itself
            // (the first fused call builds the stream of every live env, final ones included: the policy reads all of the tile's rows)
            if (KIND == QG_ENV_PAULI_NETWORK && (enabled || (fused && !resident))) {
                // PauliNetwork picks its qubit permutation here (pauli.rs:653-665)
                int perm_idx = c.nperms > 0 ? (int)(pr.misc & 0xFFFFu) : 0;
                if (c.nperms > 0 && enabled && (a.obs || a.obs_bits || fused)) {
                    const uint32_t raw = a.perm_raw ? a.perm_raw[(size_t)t * a.in_stride + env] : philox_draw(seed_of(c), (uint64_t)(c.first_id + env), tick, STREAM_PERM);
                    perm_idx = (int)__umulhi(raw, (uint32_t)c.nperms);
                    pr.misc = (pr.misc & 0xFFFF0000u) | (uint32_t)perm_idx;
                    dirty = true;
                }
                if (a.obs || a.obs_bits || fused) pn_build_obs(c, S, pr, Ob, perm_idx);
            }
            if (KIND == QG_ENV_PERMUTATION && c.OW > 0 && (enabled || (fused && !resident)) && ((a.obs && !use_cat) || a.obs_bits || fused)) {
                // one-hot rows: bit i*n + state[i] (permutation.rs:241-243)
                if (oh_full) {
                    for (int w = 0; w < c.OW; ++w) O[w] = 0;
                    for (int i = 0, b = 0; i < c.n; ++i, b += c.n) { const int bit = b + (int)get8(S, i); O[bit >> 5] |= 1u << (bit & 31); }
                } else if (oh_q0 >= 0 && oh_q0 != oh_q1) {
                    // O still holds the stream of before the SWAP: rows q0 and q1 exchange their set columns
                    const int va = (int)get8(S, oh_q1), vb = (int)get8(S, oh_q0);      // the old entries of q0 / q1
                    auto toggle = [&](int bit) { O[bit >> 5] ^= 1u << (bit & 31); };
                    toggle(oh_q0 * c.n + va); toggle(oh_q1 * c.n + vb); toggle(oh_q0 * c.n + vb); toggle(oh_q1 * c.n + va);
                }
            }
        }
        __syncwarp();
        const uint32_t mask_bits = __ballot_sync(0xFFFFFFFFu, live && !success);     // masks() = [!success; A] (clifford.rs:349-351)
        const uint32_t en_bits = __ballot_sync(0xFFFFFFFFu, live && enabled);
        if (MODE == MODE_SEARCH && a.num_active && lane == 0 && en_bits) atomicAdd(a.num_active, __popc(en_bits));
        if (MODE == MODE_STEP && a.done_bits) {
            // packed flags: lane (t % 32) keeps this step's two ballots; every 32 steps (and after the last one) the warp writes them as one
            // coalesced line per plane: done_bits[tile][bits_t0 + t]
            const uint32_t db = __ballot_sync(0xFFFFFFFFu, live && enabled && (depth == 0 || success));
            const uint32_t sb = __ballot_sync(0xFFFFFFFFu, live && enabled && success);
            if (lane == (t & 31)) { acc_done = db; acc_succ = sb; }
            if ((t & 31) == 31 || t + 1 == a.nsteps) {
                const int tl = (t & ~31) + lane;
                if (tl <= t) {
                    const size_t k = (size_t)(e0 >> 5) * (size_t)a.bits_stride + (size_t)(a.bits_t0 + tl);
                    if (EPW == 32) {
                        a.done_bits[k] = acc_done;
                        if (a.success_bits) a.success_bits[k] = acc_succ;
                    } else {                         // 16-env tiles: this tile's half of the 32-env word
                        const size_t h = 2 * k + (size_t)((e0 >> 4) & 1);
                        reinterpret_cast<uint16_t*>(a.done_bits)[h] = (uint16_t)acc_done;
                        if (a.success_bits) reinterpret_cast<uint16_t*>(a.success_bits)[h] = (uint16_t)acc_succ;
                    }
                }
            }
        }

        if constexpr (role == 1) {
            // step warp of a pair: hand the observation bits and the mask ballot over, then go on with the next step
            if (KIND == QG_ENV_PERMUTATION) cat_onehot(c, S, hand, (uint32_t)cnt, live, lane);          // (pairs need the concatenated stream for Permutation)
            else if (KIND != QG_ENV_PAULI_NETWORK) { if (live) for (int w = 0; w < c.SW; ++w) hand[w * kStride + lane] = S[w]; }
            if (lane == 0) pair_hdr[t & 1] = mask_bits;
            pair_arrive(pair_bar, t & 1, lane);
            last_en_bits = en_bits;
            continue;
        }
        // ---------------- phase 2: the warp expands its 32 environments: bits -> float observation slab, mask slab --------
        if (a.obs) {
            float* out = a.obs + ((size_t)slot * c.B + (size_t)e0) * c.obs_size;
            if (use_cat) {
                if (KIND == QG_ENV_PERMUTATION) cat_onehot(c, S, cat, (uint32_t)cnt, live, lane);
                else cat_gather<kStride>(obs_bits, cat, (uint32_t)cnt, (uint32_t)c.obs_size, a.magic_obs, lane);
                if (a.nsteps > 1) expand_cat<true>(cat, lut, out, (uint32_t)cnt * (uint32_t)c.obs_size, lane);
                else expand_cat<false>(cat, lut, out, (uint32_t)cnt * (uint32_t)c.obs_size, lane);
            } else if (KIND != QG_ENV_PERMUTATION || c.OW > 0) expand_obs<MODE, kStride>(obs_bits, lut, out, (uint32_t)cnt, (uint32_t)c.obs_size, en_bits, lane, a.magic_vpe, a.magic_obs, a.exp_q, a.exp_r, a.nsteps > 1);
            else {
                // large Permutation (no room for a bit stream in shared memory): one-hot test straight from the packed bytes
                const uint32_t total = (uint32_t)cnt * (uint32_t)c.obs_size, n = (uint32_t)c.n;
                const uint32_t* st = wbase + c.off_state * kStride;
                for (uint32_t f = lane; f < total; f += 32) {
                    const uint32_t e = fastdiv40(f, a.magic_obs), off = f - e * (uint32_t)c.obs_size;
                    const uint32_t i = __umulhi(off, c.magic_n), col = off - i * n;
                    if (MODE != MODE_SEARCH || ((en_bits >> e) & 1u)) out[f] = (((st[(i >> 2) * kStride + e] >> ((i & 3u) * 8u)) & 0xFFu) == col) ? 1.0f : 0.0f;
                }
            }
        }
        if (a.obs_bits) {
            // packed observation: the warp's 32 x OWp words are contiguous in the [B][OWp] tensor; transposed out of the
            // [word][env] shared-memory stream with coalesced stores
            const uint32_t OWp = ((uint32_t)c.obs_size + 31u) >> 5, total = (uint32_t)cnt * OWp;
            uint32_t* out = a.obs_bits + ((size_t)slot * c.B + (size_t)e0) * OWp;
            for (uint32_t i = lane; i < total; i += 32) {
                const uint32_t e = fastdiv40(i, a.magic_ow), w = i - e * OWp;
                if (MODE != MODE_SEARCH || ((en_bits >> e) & 1u)) out[i] = obs_bits[w * kStride + e];
            }
        }
        if (a.mask) {
            uint8_t* out = a.mask + ((size_t)slot * c.B + (size_t)e0) * c.A;
            if ((c.A & 3) == 0) expand_mask<MODE, 4>(out, (uint32_t)cnt, (uint32_t)c.A, mask_bits, en_bits, lane, a.magic_A);
            else expand_mask<MODE, 1>(out, (uint32_t)cnt, (uint32_t)c.A, mask_bits, en_bits, lane, a.magic_A);
        }
        if (++slot == a.ring) slot = 0;
        last_en_bits = en_bits;
        __syncwarp();                                 // the next step's phase 1 rewrites the bits phase 2 just read
    }

    if (live && dirty) {
        R[HD_DEPTH] = depth; R[HD_FLAGS] = flags; R[HD_TICK] = tick;
        if (KIND == QG_ENV_PAULI_NETWORK) { X[PX_PLO] = pr.plo; X[PX_PHI] = pr.phi; X[PX_ALIVE] = pr.alive; X[PX_ORD0] = pr.ord0; X[PX_ORD1] = pr.ord1; X[PX_MISC] = pr.misc; }
        if (MODE != MODE_OBSERVE) {
            if (!fused) {
                uint32_t* dst = c.rec + (a.dst_slot ? (int64_t)a.dst_slot[env] : env);
#pragma unroll 4
                for (int w = 0; w < c.W; ++w, dst += c.Bpad) *dst = R[w];
            }
        } else if (KIND == QG_ENV_PAULI_NETWORK) {
            c.rec[(size_t)(c.off_extra + PX_MISC) * c.Bpad + env] = pr.misc;
        }
    }
    return last_en_bits;
}

// The records of a tile that step_tile kept in shared memory (fused calls) go back to global memory.
__device__ __forceinline__ void tile_writeback(const DevCfg& c, const uint32_t* const wbase, const int lane, const int64_t e0, const int cnt) {
    if (lane >= cnt) return;
    uint32_t* dst = c.rec + e0 + lane;
    const uint32_t* src = wbase + lane;
#pragma unroll 4
    for (int w = 0; w < c.W; ++w, dst += c.Bpad, src += kStride) *dst = *src;
}

// INV: register bucket of the add_inverts inverse (qg_gf2.cuh): 0 = generic shared-memory Gauss-Jordan (or no inverts),
// 8 / 16 / 32 = matrix dimension bound of the register-resident versions.
template <int KIND, int MODE, int INV, int EPW, int PAIR = 0>
__global__ void __launch_bounds__(kWarpsPerCta * 32, INV == 32 ? 8 : 16) k_step(const __grid_constant__ DevCfg c, const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (a.pdl_mode == 1) pdl_launch_dependents();
    constexpr bool pair = PAIR != 0;                 // one tile per CTA, warp 0 steps, warp 1 stores (step_tile roles 1 / 2)
    const int64_t e0 = pair ? (int64_t)blockIdx.x * EPW : ((int64_t)blockIdx.x * kWarpsPerCta + warp) * EPW;
    if (e0 >= c.B) return;                           // whole warp leaves; no block barrier below
    const int cnt = (int)min((int64_t)EPW, c.B - e0);
    uint32_t* const wbase = smem + kLutWords + (pair ? 0 : (size_t)warp * a.sm_warp_words);
    const uint32_t* const lut = smem;                // nibble -> float4 table, first kLutWords words of the CTA's shared memory
    if (a.obs) lut_fill(smem, lane);
    if (a.pdl_mode) pdl_wait();                      // the previous grid of the stream wrote the records
    if (a.pdl_mode == 2) pdl_launch_dependents();
    if (a.stagger_ns > 0) {
        const long long wait_ns = (long long)(((int)blockIdx.x / a.num_sms) * kWarpsPerCta + warp) * a.stagger_ns;
        long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 >= wait_ns) break;
            __nanosleep(200);
        }
    }
    if constexpr (pair) {
#ifdef QG_PAIR_MBARRIER
        if (threadIdx.x == 0) {
            uint64_t* bars = reinterpret_cast<uint64_t*>(wbase + a.sm_pair_bar);
            for (int i = 0; i < 4; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"((uint32_t)__cvta_generic_to_shared(bars + i)) : "memory");
        }
        __syncthreads();                             // (both warps of a pair CTA are alive here: they share e0)
#endif
        // (which warp of the CTA steps alternates with the CTA index, so that the issue-heavy step warps do not all sit on the same
        // scheduler if warps are assigned to the SM's sub-partitions by their index within the CTA)
        const bool steps = warp == (int)(blockIdx.x & 1u);
        if (steps) step_tile<KIND, MODE, INV, EPW, 1>(c, a, wbase, lut, lane, e0, cnt);
        else step_tile<KIND, MODE, INV, EPW, 2>(c, a, wbase, lut, lane, e0, cnt);
    } else {
        step_tile<KIND, MODE, INV, EPW, 0>(c, a, wbase, lut, lane, e0, cnt);
    }
}

// ---- load (set_state / constructor) --------------------------------------------------------------
// staged: payloads of PW words = state words (+ PauliNetwork extras); env first + i reads payload i / group (group = 1: one payload per
// env; group = count: every env reads payload 0; qg_set_state_grouped: one payload per group of rollouts).
template <int KIND>
__global__ void k_load(const __grid_constant__ DevCfg c, const uint32_t* __restrict__ staged, int PW, int64_t first, int64_t count, int64_t group, uint32_t depth_init) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t env = first + i;
    const uint32_t* src = staged + (size_t)(i / group) * PW;
    auto put = [&](int w, uint32_t v) { c.rec[(size_t)w * c.Bpad + env] = v; };
    bool ok = true;
    if (KIND == QG_ENV_PERMUTATION) {
        for (int q = 0; q < c.n; ++q) if (((src[q >> 2] >> ((q & 3) * 8)) & 0xFFu) != (uint32_t)q) ok = false;
    } else if (KIND == QG_ENV_PAULI_NETWORK) {
        ok = (src[PW - 1] & 1u) != 0;      // PauliNetwork::solved precomputed by the host packer (last staged word)
    } else {
        for (int w = 0; w < c.SW; ++w) if (src[w] != c.ident[w]) ok = false;
    }
    for (int w = 0; w < c.SW; ++w) put(c.off_state + w, src[w]);
    if (KIND == QG_ENV_PAULI_NETWORK) {
        const int XW = PW - c.SW - 1;
        for (int w = 0; w < XW; ++w) put(c.off_extra + w, src[c.SW + w]);
    }
    for (int w = 0; w < c.MW; ++w) { put(c.off_lastg + w, 0xFFFFFFFFu); put(c.off_lastcx + w, 0xFFFFFFFFu); }
    put(HD_DEPTH, depth_init);
    put(HD_FLAGS, ok ? FL_SUCCESS : 0u);
    put(HD_NCNOTS, 0); put(HD_NGATES, 0); put(HD_LAYERS, 0);
    put(HD_REWARD, __float_as_uint(ok ? 1.0f : 0.0f));
    put(HD_TICK, 0);
}

// ---- read-out of a search (k_best, k_best_grouped, k_solutions, k_pack_winner) ------------------------------------------------------
// key = success<<62 | orderable_u32(return)<<30 | (2^30-1 - global rollout id): the largest key is the best rollout
__device__ __forceinline__ unsigned long long rollout_key(bool success, float ret, int64_t gid) {
    uint32_t u = __float_as_uint(ret);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);      // order-preserving map f32 -> u32
    return ((unsigned long long)(success ? 1 : 0) << 62) | ((unsigned long long)u << 30) | (unsigned long long)((0x3FFFFFFFll - gid) & 0x3FFFFFFFll);
}
// Env::solution of `env` (its n logged entries) into row[0..n): the column of the slot-major log sol[slot][env], entries logged while the
// env was inverted (bit 31: LinearFunction / Clifford / Permutation) after the others, in reverse order (clifford.rs:376-381); PauliNetwork
// words as logged (bit 31 there is ROTATION_MARKER, pauli.rs:685-719).
__device__ __forceinline__ void write_solution(const DevCfg& c, int64_t env, int n, uint32_t* __restrict__ row) {
    const uint32_t* col = c.sol + env;
    if (c.kind == QG_ENV_PAULI_NETWORK) {
        for (int k = 0; k < n; ++k) row[k] = col[(size_t)k * c.Bpad];
        return;
    }
    int w = 0;
    for (int k = 0; k < n; ++k) { const uint32_t v = col[(size_t)k * c.Bpad]; if (!(v & 0x80000000u)) row[w++] = v; }
    for (int k = n - 1; k >= 0; --k) { const uint32_t v = col[(size_t)k * c.Bpad]; if (v & 0x80000000u) row[w++] = v & 0x7FFFFFFFu; }
}

// ---- reset (Permutation / LinearFunction / Clifford): identity scrambled by `difficulty` Philox-drawn gates
// (permutation.rs:175-192, linear_function.rs:285-300, clifford.rs:306-319) --------------------------
// which environments a reset touches: RESET_ALL, RESET_FINAL (those whose is_final() holds: what a collector does between
// episodes) or RESET_SELECT (select[env] != 0)
enum { RESET_ALL = 0, RESET_FINAL = 1, RESET_SELECT = 2 };
__device__ __forceinline__ bool reset_wanted(const DevCfg& c, int64_t env, int which, const uint8_t* select) {
    if (which == RESET_SELECT) return select[env] != 0;
    if (which == RESET_FINAL) return c.rec[(size_t)HD_DEPTH * c.Bpad + env] == 0 || (c.rec[(size_t)HD_FLAGS * c.Bpad + env] & FL_SUCCESS) != 0;
    return true;
}

template <int KIND, int EPC>
__global__ void __launch_bounds__(EPC) k_reset(const __grid_constant__ DevCfg c, int which, const uint8_t* __restrict__ select) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * EPC + tid;
    if (env >= c.B) return;
    if (!reset_wanted(c, env, which, select)) return;
    typedef SmWords<EPC> Wd;
    const Wd S{smem + tid};
    if (KIND == QG_ENV_PERMUTATION) { for (int w = 0; w < c.SW; ++w) S[w] = 0; for (int q = 0; q < c.n; ++q) set8(S, q, (uint32_t)q); }
    else for (int w = 0; w < c.SW; ++w) S[w] = c.ident[w];
    const uint64_t seed = seed_of(c);
    for (int k = 0; k < c.difficulty; ++k) {
        const uint32_t raw = philox_draw(seed, (uint64_t)(c.first_id + env), (uint32_t)k, STREAM_RESET);
        const int act = (int)__umulhi(raw, (uint32_t)c.A);      // Uniform::new(0, num_actions)
        const uint32_t g = __ldg(c.gates + act);
        apply_gate_state<KIND>(c, S, (int)(g & 0xFFu), (int)((g >> 8) & 0xFFu), (int)((g >> 16) & 0xFFu));
    }
    const bool ok = solved_state<KIND>(c, S);
    auto put = [&](int w, uint32_t v) { c.rec[(size_t)w * c.Bpad + env] = v; };
    for (int w = 0; w < c.SW; ++w) put(c.off_state + w, S[w]);
    for (int w = 0; w < c.MW; ++w) { put(c.off_lastg + w, 0xFFFFFFFFu); put(c.off_lastcx + w, 0xFFFFFFFFu); }
    const long long d = (long long)c.depth_slope * (long long)c.difficulty;
    put(HD_DEPTH, (uint32_t)(d < (long long)c.max_depth ? d : (long long)c.max_depth));
    put(HD_FLAGS, ok ? FL_SUCCESS : 0u);
    put(HD_NCNOTS, 0); put(HD_NGATES, 0); put(HD_LAYERS, 0);
    put(HD_REWARD, __float_as_uint(ok ? 1.0f : 0.0f));
    put(HD_TICK, 0);
    c.ret[env] = 0.0f;
}

// ---- PauliNetwork reset (pauli.rs:554-586): rotations from generate_paulis_with_difficulty (115-213), tableau from
// random_clifford_tableau (220-271), then the initial clean.  All draws come from one Philox stream per env
// (draw index = running counter), in the order the reference code makes them.
// gen tables (c.pgen): [0]=ND, [1]=NP, [2]=NCX, dists[ND] ascending, pair_off[ND+1], pairs[NP] (q1 | q2<<8, q1<q2), cx[NCX] (q0 | q1<<8)
template <int EPC>
__global__ void __launch_bounds__(EPC) k_reset_pauli(const __grid_constant__ DevCfg c, int pauli_diff_scale, float decay, int final_layers, int which,
                                                      const uint8_t* __restrict__ select) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x;
    const int64_t env = (int64_t)blockIdx.x * EPC + tid;
    if (env >= c.B) return;
    if (!reset_wanted(c, env, which, select)) return;
    typedef SmWords<EPC> Wd;
    const Wd S{smem + tid}, X = S.at(c.SW), RX = X.at(c.W - c.off_extra), RZ = RX.at(c.Rtot), HV = RZ.at(c.Rtot);
    const int n = c.n, D = 2 * n;
    const uint32_t* tab = c.pgen;
    const int ND = (int)tab[0], NCX = (int)tab[2];
    const uint32_t* dists = tab + 3; const uint32_t* poff = dists + ND; const uint32_t* pairs = poff + ND + 1; const uint32_t* cxp = pairs + tab[1];
    uint32_t ctr = 0;
    const uint64_t seed = seed_of(c);
    auto draw = [&]() { return philox_draw(seed, (uint64_t)(c.first_id + env), ctr++, STREAM_RESET); };
    auto below = [&](uint32_t k) { return __umulhi(draw(), k); };
    auto unit = [&]() { return (float)(draw() >> 8) * (1.0f / 16777216.0f); };
    auto count_le = [&](uint32_t lim) { int k = 0; while (k < ND && dists[k] <= lim) ++k; return k; };

    // --- rotations
    int R = 0;
    uint32_t remaining = (uint32_t)c.difficulty / (uint32_t)pauli_diff_scale;
    while (remaining > 0 && R < final_layers) {
        const uint32_t diff = remaining;
        const int nvalid = count_le(diff);
        if (nvalid == 0) break;
        uint32_t qubits = 0, pd = diff;
        uint32_t nd = below((uint32_t)nvalid);
        uint32_t pr = pairs[poff[nd] + below(poff[nd + 1] - poff[nd])];
        qubits |= (1u << (pr & 0xFFu)) | (1u << (pr >> 8));
        pd = pd > dists[nd] ? pd - dists[nd] : 0u;
        for (;;) {
            const int nvd = min(count_le(pd), nvalid);
            if (pd == 0 || nvd == 0 || __popc(qubits) >= n) break;
            if (unit() <= decay) break;
            nd = below((uint32_t)nvd);
            uint32_t nvp = 0;
            for (uint32_t i = poff[nd]; i < poff[nd + 1]; ++i) { const uint32_t q = pairs[i]; if (((qubits >> (q & 0xFFu)) | (qubits >> (q >> 8))) & 1u) ++nvp; }
            if (nvp == 0) continue;
            uint32_t pick = below(nvp);
            for (uint32_t i = poff[nd]; i < poff[nd + 1]; ++i) {
                const uint32_t q = pairs[i];
                if (((qubits >> (q & 0xFFu)) | (qubits >> (q >> 8))) & 1u) { if (pick == 0) { pr = q; break; } --pick; }
            }
            qubits |= (1u << (pr & 0xFFu)) | (1u << (pr >> 8));
            pd = pd > dists[nd] ? pd - dists[nd] : 0u;
        }
        uint32_t x = 0, z = 0;
        // the label string holds qubit q's axis at string position q, and Pauli::from_label reads position p as
        // qubit n-1-p (pauli.rs:62), so the generated axis lands on qubit n-1-q.
        for (int q = 0; q < n; ++q) if ((qubits >> q) & 1u) { const uint32_t ax = below(3u); const int k = n - 1 - q; if (ax != 2u) x |= 1u << k; if (ax != 0u) z |= 1u << k; }
        RX[R] = x; RZ[R] = z; ++R;
        const uint32_t cost = max(diff - pd, 1u);
        remaining = remaining > cost ? remaining - cost : 0u;
    }
    // --- tableau
    for (int w = 0; w < c.SW; ++w) S[w] = 0;
    for (int r = 0; r < D; ++r) xor_bits(S, r * c.CW + r, 1, 1u);
    if (c.difficulty != 0 && NCX != 0) {
        for (int k = 0; k < c.difficulty; ++k) {
            const float r = unit();
            if (r > 0.3f) { const uint32_t pr = cxp[below((uint32_t)NCX)]; const int q0 = (int)(pr & 0xFFu), q1 = (int)(pr >> 8); row_xor(S, c.CW, q1, q0); row_xor(S, c.CW, n + q0, n + q1); }
            else if (r > 0.15f) { const int q = (int)below((uint32_t)n); row_swap(S, c.CW, q, n + q); }
            else { const int q = (int)below((uint32_t)n); row_xor(S, c.CW, n + q, q); }
        }
    }
    // --- attach rotations: columns, phases (#Y mod 4), anticommutation rows
    for (int w = 0; w < c.W - c.off_extra; ++w) X[w] = 0;
    PauliRegs p{}; p.ord0 = 0x76543210u; p.ord1 = 0xFEDCBA98u;
    for (int r = 0; r < R; ++r) {
        const uint32_t x = RX[r], z = RZ[r];
        for (int q = 0; q < n; ++q) { if ((x >> q) & 1u) xor_bits(S, q * c.CW + D + r, 1, 1u); if ((z >> q) & 1u) xor_bits(S, (n + q) * c.CW + D + r, 1, 1u); }
        const uint32_t ys = (uint32_t)__popc(x & z) & 3u;
        p.plo |= (ys & 1u) << r; p.phi |= (ys >> 1) << r;
        uint32_t anti = 0;
        for (int j = 0; j < r; ++j) if ((__popc(x & RZ[j]) + __popc(z & RX[j])) & 1) anti |= 1u << j;
        X[PX_ANTI + (r >> 1)] |= anti << ((r & 1) * 16);
    }
    p.alive = (R >= 32) ? 0xFFFFFFFFu : ((1u << R) - 1u);
    p.misc = ((uint32_t)R << 16) | ((uint32_t)R << 24);
    int nh = 0; uint32_t err = 0;
    pn_clean(c, S, X, p, HV, nh, err);                      // "clean initially trivial rotations" (pauli.rs:575)
    const bool ok = pn_solved(c, S, p);
    X[PX_PLO] = p.plo; X[PX_PHI] = p.phi; X[PX_ALIVE] = p.alive; X[PX_ORD0] = p.ord0; X[PX_ORD1] = p.ord1; X[PX_MISC] = p.misc;
    auto put = [&](int w, uint32_t v) { c.rec[(size_t)w * c.Bpad + env] = v; };
    for (int w = 0; w < c.SW; ++w) put(c.off_state + w, S[w]);
    for (int w = 0; w < c.W - c.off_extra; ++w) put(c.off_extra + w, X[w]);
    for (int w = 0; w < c.MW; ++w) { put(c.off_lastg + w, 0xFFFFFFFFu); put(c.off_lastcx + w, 0xFFFFFFFFu); }
    const long long d = (long long)c.depth_slope * (long long)c.difficulty;
    put(HD_DEPTH, (uint32_t)(d < (long long)c.max_depth ? d : (long long)c.max_depth));
    put(HD_FLAGS, (ok ? FL_SUCCESS : 0u) | (err << FL_ERR_SHIFT));
    put(HD_NCNOTS, 0); put(HD_NGATES, 0); put(HD_LAYERS, 0);
    put(HD_REWARD, __float_as_uint(ok ? 1.0f : 0.0f));
    put(HD_TICK, 0);
    c.ret[env] = 0.0f;
}

}  // namespace qg
