// qg_mcts.cu — batched PUCT tree search on the device (SURVEY.md §8f row 4; `num_mcts_searches > 0` in the reference's
// `algorithm.solve(state, deterministic, num_searches, num_mcts_searches, C, max_expand_depth)`, rl/synthesis.py:122-124,
// rl/configs.py:30-42).  twisterl's own MCTS is not in the reference tree, so the protocol below is this engine's, stated
// here and restated on the CPU in tests/test_mcts.py (parity of the search itself is unpinned, SURVEY.md §8c):
//
//   one tree per rollout, rebuilt for every decision; node 0 = the rollout's current env state.  A node stores, per action a,
//   the policy prior P(a), the visit count N(a), the sum W(a) of the returns backed up through the edge and the child node
//   (or -1); plus the reward of the step that created it and whether its env is final.
//   simulation:  descend from the root taking  argmax_a  W(a)/N(a) [0 if N(a) = 0]  +  C * P(a) * sqrt(1 + sum_b N(b)) / (1 + N(a))
//                (lowest a on ties) until the edge has no child (the child is then created by cloning the parent's env record
//                and stepping it: qg_step_slots) or the node reached is final;
//                the new node gets the policy's priors for its observation; its value v is the value head's output, 0 if final;
//                back up  G <- reward(child) + G  from the leaf (G = v) to the root, N(a) += 1, W(a) += G on every edge.
//   decision:    action weights = N(a) / sum N at the root (arg-max or Philox sample by qg_search_step).
//   tree reuse (opt-in, MCTSSearch(reuse_tree=True); node_cap = 2S + 1 for S simulations per decision): after the rollouts' step,
//                tree i is re-rooted (qg_mcts_reroot) when the rollout played an action a >= 0 (chosen[i]), the root has a child
//                c = child[0][a], and the pool record of c equals the rollout's record word for word (the solution-log length of
//                HD_FLAGS masked as k_copy_records masks it).  With add_inverts the pool and the rollout draw their own coins, so c is one
//                sample of a stochastic step: the record test keeps it only when the rollout reached the same env.  A re-rooted tree
//                keeps the first K = node_cap - S nodes of c's subtree in creation order (a prefix in creation order holds every kept
//                node's parent), renumbered in that order so that c becomes node 0; prior, N, W, remapped children, reward, final flag
//                and pool record move with each node.  An edge whose child was dropped keeps N and W and gets child = -1.  The root keeps
//                its stored prior (qg_mcts_begin_keep skips it); every other tree starts fresh.  The decision then adds S simulations.
// Every f32 operation is rounded on its own (no FMA contraction) so the CPU restatement reproduces each argmax.
//
// Decomposition: one warp per tree; lanes stride over the actions of a node for the PUCT arg-max and for initialising a
// new node's arrays; the walk itself is sequential per tree.  Trees are independent: no cross-warp communication.
#include <algorithm>
#include <string>

#include "qg_engine_priv.hpp"

namespace qg {

__device__ __forceinline__ void warp_argmax(float& s, int& a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float so = __shfl_xor_sync(0xFFFFFFFFu, s, o);
        const int ao = __shfl_xor_sync(0xFFFFFFFFu, a, o);
        if (so > s || (so == s && ao < a)) { s = so; a = ao; }
    }
}

__device__ __forceinline__ void begin_tree(const qg_mcts_tree& t, int tree, int lane, const float* __restrict__ root_prior, const uint8_t* __restrict__ root_final) {
    const size_t base = (size_t)tree * t.node_cap;
    for (int a = lane; a < t.num_actions; a += 32) {
        const size_t k = base * t.num_actions + a;
        t.prior[k] = root_prior[(size_t)tree * t.num_actions + a];
        t.visits[k] = 0; t.value_sum[k] = 0.0f; t.child[k] = -1;
    }
    if (lane == 0) { t.node_count[tree] = 1; t.node_reward[base] = 0.0f; t.node_final[base] = root_final[tree] ? 1 : 0; t.path_len[tree] = 0; t.new_node[tree] = -1; }
}

__global__ void k_mcts_begin(const qg_mcts_tree t, const float* __restrict__ root_prior, const uint8_t* __restrict__ root_final) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees) return;
    begin_tree(t, tree, lane, root_prior, root_final);
}

__global__ void k_mcts_begin_keep(const qg_mcts_tree t, const float* __restrict__ root_prior, const uint8_t* __restrict__ root_final,
                                  const uint8_t* __restrict__ reused) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees || reused[tree]) return;
    begin_tree(t, tree, lane, root_prior, root_final);
}

// Re-rooting (protocol above).  path_node of tree i holds the old -> new node id map: >= 0 kept under that id, -2 a member of c's subtree
// that is not kept (yet), -1 not a member.  Pass 1 walks nodes c .. node_count-1 in creation order; a member takes the next new id and marks
// its children, so a node's mark is final before the walk reaches it (children are created after their parent).  Pass 2 moves the kept
// nodes in ascending old-id order in place: new id <= old id and every lane moves the same entries of every row, so no row is written
// before it has been read.
__global__ void k_mcts_reroot(const qg_mcts_tree t, uint32_t* pool_rec, int64_t pool_bpad, const uint32_t* __restrict__ roll_rec, int64_t roll_bpad,
                              int W, const int32_t* __restrict__ chosen, int keep, uint8_t* __restrict__ reused) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees) return;
    const size_t base = (size_t)tree * t.node_cap;
    const int A = t.num_actions, a = chosen[tree];
    const int c = (a >= 0 && a < A) ? t.child[base * A + a] : -1;
    bool diff = c < 0;
    if (c >= 0) {
        const uint32_t len_mask = (1u << FL_LEN_SHIFT) - 1u;
        for (int w = lane; w < W; w += 32) {
            const uint32_t m = w == HD_FLAGS ? len_mask : 0xFFFFFFFFu;
            diff |= ((pool_rec[(size_t)w * pool_bpad + base + c] ^ roll_rec[(size_t)w * roll_bpad + tree]) & m) != 0u;
        }
    }
    diff = __any_sync(0xFFFFFFFFu, diff);
    if (lane == 0) reused[tree] = diff ? 0 : 1;
    if (diff) return;
    volatile int32_t* map = t.path_node + base;
    const int count = t.node_count[tree];
    for (int j = c + lane; j < count; j += 32) map[j] = -1;
    __syncwarp();
    int kept = 0;
    for (int j = c; j < count && kept < keep; ++j) {
        if (j != c && map[j] == -1) continue;
        if (lane == 0) map[j] = kept;
        ++kept;
        for (int b = lane; b < A; b += 32) {
            const int ch = t.child[(base + j) * A + b];
            if (ch >= 0) map[ch] = -2;
        }
        __syncwarp();
    }
    for (int j = c, moved = 0; moved < kept; ++j) {
        const int nj = map[j];
        if (nj < 0) continue;
        ++moved;
        const size_t src = (base + j) * A, dst = (base + nj) * A;
        for (int b = lane; b < A; b += 32) {
            const int ch = t.child[src + b];
            const int nc = ch >= 0 ? map[ch] : -1;
            const float p = t.prior[src + b], s = t.value_sum[src + b];
            const int n = t.visits[src + b];
            t.prior[dst + b] = p; t.visits[dst + b] = n; t.value_sum[dst + b] = s; t.child[dst + b] = nc >= 0 ? nc : -1;
        }
        for (int w = lane; w < W; w += 32) pool_rec[(size_t)w * pool_bpad + base + nj] = pool_rec[(size_t)w * pool_bpad + base + j];
        if (lane == 0) { t.node_reward[base + nj] = t.node_reward[base + j]; t.node_final[base + nj] = t.node_final[base + j]; }
    }
    if (lane == 0) t.node_count[tree] = kept;
}

__global__ void k_mcts_select(const qg_mcts_tree t, float c_puct, int32_t* __restrict__ src_slot, int32_t* __restrict__ dst_slot, int32_t* __restrict__ action) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees) return;
    const size_t base = (size_t)tree * t.node_cap;
    const int A = t.num_actions;
    int node = 0, len = 0, act = -1, newn = -1, src = 0;
    if (!t.node_final[base]) {
        for (;;) {
            const size_t row = (base + node) * A;
            int tot = 0;
            for (int a = lane; a < A; a += 32) tot += t.visits[row + a];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xFFFFFFFFu, tot, o);
            const float sq = sqrtf((float)(tot + 1));
            float best = -INFINITY; int besta = 0x7FFFFFFF;
            for (int a = lane; a < A; a += 32) {
                const int n = t.visits[row + a];
                const float q = n > 0 ? __fdiv_rn(t.value_sum[row + a], (float)n) : 0.0f;
                const float u = __fdiv_rn(__fmul_rn(__fmul_rn(c_puct, t.prior[row + a]), sq), (float)(n + 1));
                const float s = __fadd_rn(q, u);
                if (s > best || (s == best && a < besta)) { best = s; besta = a; }
            }
            warp_argmax(best, besta);
            if (besta >= A) besta = 0;                       // every score was NaN: fall back to action 0
            if (lane == 0) { t.path_node[base + len] = node; t.path_action[base + len] = besta; }
            ++len;
            int c = 0;
            if (lane == 0) {                                 // lane 0 owns the tree's bookkeeping; the others follow its decision
                c = t.child[row + besta];
                if (c < 0) { newn = t.node_count[tree]; t.child[row + besta] = newn; t.node_count[tree] = newn + 1; }
            }
            c = __shfl_sync(0xFFFFFFFFu, c, 0);
            if (c < 0) {
                newn = __shfl_sync(0xFFFFFFFFu, newn, 0);
                src = node; act = besta;
                break;
            }
            node = c;
            if (t.node_final[base + node] || len >= t.node_cap) break;      // revisit of a final node: nothing to expand
        }
    }
    __syncwarp();
    if (lane == 0) {
        src_slot[tree] = (int32_t)(base + src);
        dst_slot[tree] = (int32_t)(base + (newn >= 0 ? newn : 0));
        action[tree] = act;
        t.path_len[tree] = len; t.new_node[tree] = newn;
    }
}

__global__ void k_mcts_backup(const qg_mcts_tree t, const float* __restrict__ prior_in, const float* __restrict__ value_in,
                              const float* __restrict__ reward_in, const uint8_t* __restrict__ done_in) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees) return;
    const size_t base = (size_t)tree * t.node_cap;
    const int A = t.num_actions, len = t.path_len[tree], newn = t.new_node[tree];
    float v = 0.0f;
    if (newn >= 0) {
        const size_t row = (base + newn) * A;
        for (int a = lane; a < A; a += 32) {
            t.prior[row + a] = prior_in[(size_t)tree * A + a];
            t.visits[row + a] = 0; t.value_sum[row + a] = 0.0f; t.child[row + a] = -1;
        }
        const bool fin = done_in[tree] != 0;
        if (lane == 0) { t.node_reward[base + newn] = reward_in[tree]; t.node_final[base + newn] = fin ? 1 : 0; }
        v = fin ? 0.0f : value_in[tree];
    }
    __syncwarp();
    if (lane == 0) {
        float G = v;
        for (int i = len - 1; i >= 0; --i) {
            const size_t k = (base + t.path_node[base + i]) * A + t.path_action[base + i];
            G = __fadd_rn(t.node_reward[base + t.child[k]], G);
            t.visits[k] += 1;
            t.value_sum[k] = __fadd_rn(t.value_sum[k], G);
        }
    }
}

__global__ void k_mcts_root_weights(const qg_mcts_tree t, float* __restrict__ weights) {
    const int tree = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (tree >= t.num_trees) return;
    const size_t row = (size_t)tree * t.node_cap * t.num_actions;
    int tot = 0;
    for (int a = lane; a < t.num_actions; a += 32) tot += t.visits[row + a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xFFFFFFFFu, tot, o);
    for (int a = lane; a < t.num_actions; a += 32) weights[(size_t)tree * t.num_actions + a] = tot > 0 ? __fdiv_rn((float)t.visits[row + a], (float)tot) : 0.0f;
}

static int check_tree(const qg_mcts_tree* t) {
    if (!t || t->num_trees < 0 || t->node_cap < 1 || t->num_actions < 1) { set_error("qg_mcts: bad tree descriptor"); return QG_ERR_INVALID; }
    if (!t->prior || !t->visits || !t->value_sum || !t->child || !t->node_reward || !t->node_final || !t->node_count || !t->path_node || !t->path_action ||
        !t->path_len || !t->new_node) { set_error("qg_mcts: null tree array"); return QG_ERR_INVALID; }
    if ((int64_t)t->num_trees * t->node_cap > 0x7FFFFFFFll) { set_error("qg_mcts: more than 2^31 node slots"); return QG_ERR_UNSUPPORTED; }
    return QG_OK;
}
static inline unsigned tree_grid(const qg_mcts_tree* t) { return (unsigned)(((int64_t)t->num_trees * 32 + 127) / 128); }

}  // namespace qg

using namespace qg;

#define MCTS_LAUNCHED()                                                                                     \
    do {                                                                                                    \
        const cudaError_t _e = cudaGetLastError();                                                          \
        if (_e != cudaSuccess) { set_error(std::string("qg_mcts launch: ") + cudaGetErrorString(_e)); return QG_ERR_CUDA; } \
    } while (0)

extern "C" {

int qg_mcts_begin(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!root_prior_dev || !root_final_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    k_mcts_begin<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, root_prior_dev, root_final_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

int qg_mcts_select(const qg_mcts_tree* t, float c_puct, int32_t* src_slot_dev, int32_t* dst_slot_dev, int32_t* action_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!src_slot_dev || !dst_slot_dev || !action_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    k_mcts_select<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, c_puct, src_slot_dev, dst_slot_dev, action_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

int qg_mcts_backup(const qg_mcts_tree* t, const float* prior_dev, const float* value_dev, const float* reward_dev, const uint8_t* done_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!prior_dev || !value_dev || !reward_dev || !done_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    k_mcts_backup<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, prior_dev, value_dev, reward_dev, done_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

int qg_mcts_root_weights(const qg_mcts_tree* t, float* weights_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!weights_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    k_mcts_root_weights<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, weights_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

int qg_mcts_reroot(const qg_mcts_tree* t, qg_engine* pool, const qg_engine* rollouts, const int32_t* chosen_dev, int32_t keep_nodes,
                   uint8_t* reused_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!pool || !rollouts || !chosen_dev || !reused_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (pool->L.kind != rollouts->L.kind || pool->L.n != rollouts->L.n || pool->L.W != rollouts->L.W || pool->L.A != rollouts->L.A ||
        pool->device != rollouts->device || t->num_actions != pool->L.A) {
        set_error("qg_mcts_reroot: the engines must share env kind, qubits, gateset size and device with the trees"); return QG_ERR_INVALID;
    }
    if (rollouts->B < t->num_trees || pool->B < (int64_t)t->num_trees * t->node_cap) {
        set_error("qg_mcts_reroot: the rollout engine needs one env per tree and the pool node_cap slots per tree"); return QG_ERR_INVALID;
    }
    if (keep_nodes < 1 || keep_nodes > t->node_cap) { set_error("qg_mcts_reroot: keep_nodes must be in 1..node_cap"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(pool->device));
    k_mcts_reroot<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, pool->dc.rec, pool->Bpad, rollouts->dc.rec, rollouts->Bpad, pool->L.W, chosen_dev,
                                                                  keep_nodes, reused_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

int qg_mcts_begin_keep(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, const uint8_t* reused_dev, qg_stream stream) {
    const int rc = check_tree(t);
    if (rc != QG_OK) return rc;
    if (!root_prior_dev || !root_final_dev || !reused_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (t->num_trees == 0) return QG_OK;
    k_mcts_begin_keep<<<tree_grid(t), 128, 0, (cudaStream_t)stream>>>(*t, root_prior_dev, root_final_dev, reused_dev);
    MCTS_LAUNCHED();
    return QG_OK;
}

}  // extern "C"
