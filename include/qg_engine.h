/* qg_engine.h — C ABI of the B200 batched synthesis-environment engine.
 *
 * This is the drop-in boundary for qiskit-gym's one data-parallel hot path: stepping many
 * independent synthesis environments (Permutation, LinearFunction, Clifford, PauliNetwork)
 * and the synth-time rollout search.  Every entry point replaces one method of the
 * reference's `impl twisterl::rl::env::Env for X` blocks, batched over B environments.
 * Reference paths are relative to /root/reference/rust/src.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types; all functions return an int status
 *    (QG_OK = 0, negative = error; message via qg_last_error()); nothing throws.
 *  - pointers named *_dev are device pointers on the engine's GPU; *_host are host pointers.
 *  - every device entry takes a CUDA stream (`qg_stream`, a cudaStream_t), is asynchronous on
 *    that stream and allocates nothing; the *_host convenience calls synchronise the stream.
 *  - one engine is bound to one GPU and is driven by one host thread at a time.
 *  - the library fails (QG_ERR_CUDA) when no CUDA device is usable: there is no CPU fallback.
 */
#ifndef QG_ENGINE_H
#define QG_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QG_API __attribute__((visibility("default")))

typedef struct CUstream_st* qg_stream;   /* == cudaStream_t */
typedef struct qg_engine qg_engine;
typedef struct qg_twists qg_twists;

/* status codes */
enum {
    QG_OK = 0,
    QG_ERR_INVALID = -1,     /* bad argument / config (the reference raises ValueError/TypeError or panics) */
    QG_ERR_CUDA = -2,        /* CUDA runtime failure or no device */
    QG_ERR_UNSUPPORTED = -3, /* size outside the engine's limits (see qg_limits) */
    QG_ERR_STATE = -4        /* malformed set_state payload */
};

/* envs (lib.rs:24-30) */
enum { QG_ENV_PERMUTATION = 0, QG_ENV_LINEAR_FUNCTION = 1, QG_ENV_CLIFFORD = 2, QG_ENV_PAULI_NETWORK = 3 };

/* gate kinds (envs/common.rs:19-29) */
enum { QG_H = 0, QG_S = 1, QG_SDG = 2, QG_SX = 3, QG_SXDG = 4, QG_CX = 5, QG_CZ = 6, QG_SWAP = 7 };

typedef struct qg_gate { int32_t kind; int32_t q0; int32_t q1; } qg_gate;   /* q1 unused for 1-qubit gates */

/* Constructor arguments of the four pyo3 classes (permutation.rs:266-299,
 * linear_function.rs:373-406, clifford.rs:390-423, pauli.rs:728-775); `None` defaults are
 * resolved by the caller (qg_config_default does it). */
typedef struct qg_config {
    int32_t env_kind;
    int32_t num_qubits;
    int32_t difficulty;
    int32_t depth_slope;
    int32_t max_depth;
    int32_t num_gates;
    const qg_gate* gateset;
    float w_n_cnots, w_n_layers_cnots, w_n_layers, w_n_gates;   /* MetricsWeights, metrics.rs:149-184 */
    int32_t add_inverts;          /* ignored by PauliNetwork */
    int32_t add_perms;
    int32_t track_solution;
    /* PauliNetwork only */
    int32_t max_rotations;
    int32_t pauli_diff_scale;
    float num_qubits_decay;
    int32_t final_pauli_layers;
    float pauli_layer_reward;
    /* engine extras */
    int32_t solution_capacity;    /* entries kept per env; 0 = max_depth (+ rotations for Pauli) */
    int32_t tile_envs;            /* envs per warp tile of the step kernel: 0 = chosen per launch from the batch size, or 16 / 32 */
} qg_config;

/* error flag bits reported by qg_read_errors (situations where the reference panics) */
enum {
    QG_FLAG_SINGULAR = 1,        /* inverse of a singular matrix requested (linear_function.rs:131, clifford.rs:155) */
    QG_FLAG_SOLUTION_OVERFLOW = 2,
    QG_FLAG_LAYER_OVERFLOW = 4,  /* a layer counter passed 32767 */
    QG_FLAG_BAD_ROTATION = 8,    /* zero-weight rotation met by the cleaner (pauli_network.rs:114 unwrap) */
    QG_FLAG_BAD_ACTION = 16      /* negative action index */
};

/* ---- library / host-only helpers (usable without a GPU) ---------------------------------- */
QG_API const char* qg_version(void);
QG_API const char* qg_last_error(void);
/* Fills every field with the reference defaults (metrics 0.01/0/0/0.0001, add_inverts=add_perms=
 * track_solution=1, depth_slope=2, max_depth=128, difficulty=1, max_rotations=5, pauli_diff_scale=8,
 * num_qubits_decay=0.5, final_pauli_layers=-1 (=> max_rotations+2), pauli_layer_reward=0.01). */
QG_API void qg_config_default(qg_config* cfg, int32_t env_kind);
/* Gate-name parser of common.rs:46-100 (trim, case-insensitive, arity check).
 * Returns the gate kind, QG_ERR_INVALID for an unknown name, QG_ERR_STATE for a wrong arity. */
QG_API int qg_gate_kind_from_name(const char* name, int32_t num_indices);
/* Validates a config the way construction would (gate arity/indices, size limits). */
QG_API int qg_config_validate(const qg_config* cfg);
/* obs_shape() / num_actions() / set_state payload length (0 = variable, PauliNetwork) */
QG_API int qg_config_obs_shape(const qg_config* cfg, int32_t out_shape[2]);
QG_API int64_t qg_config_state_len(const qg_config* cfg);
/* twists() (symmetry.rs:297-361): obs_perms/act_perms (or raw qubit perms for PauliNetwork). */
QG_API int qg_twists_create(const qg_config* cfg, qg_twists** out);
QG_API void qg_twists_destroy(qg_twists* t);
QG_API int64_t qg_twists_count(const qg_twists* t);
QG_API int64_t qg_twists_obs_len(const qg_twists* t);   /* entries per obs perm */
QG_API int64_t qg_twists_act_len(const qg_twists* t);
QG_API int qg_twists_copy(const qg_twists* t, int64_t* obs_perms_host, int64_t* act_perms_host);
/* device memory an engine of this config and batch needs (bytes) */
QG_API int64_t qg_workspace_bytes(const qg_config* cfg, int64_t batch);

/* ---- engine lifetime ------------------------------------------------------------------- */
/* workspace_dev: caller-owned device buffer of qg_workspace_bytes() bytes (256-byte aligned), or
 * NULL to let the engine cudaMalloc it.  All envs start as the reference constructor leaves them
 * (identity, depth 1, success, reward 1.0). */
QG_API int qg_create(const qg_config* cfg, int32_t device, int64_t batch, void* workspace_dev, qg_engine** out);
QG_API void qg_destroy(qg_engine* e);
QG_API int64_t qg_batch(const qg_engine* e);
QG_API int32_t qg_num_actions(const qg_engine* e);          /* Env::num_actions */
QG_API int32_t qg_obs_size(const qg_engine* e);             /* prod(obs_shape()) */
QG_API int qg_obs_shape(const qg_engine* e, int32_t out_shape[2]);   /* Env::obs_shape */
QG_API int qg_set_difficulty(qg_engine* e, int32_t difficulty);      /* Env::set_difficulty */
QG_API int32_t qg_get_difficulty(const qg_engine* e);                /* Env::get_difficulty */

/* ---- state in ---------------------------------------------------------------------------- */
/* Env::set_state (permutation.rs:168-173, linear_function.rs:279-283, clifford.rs:299-304,
 * pauli.rs:517-552) for `count` envs starting at env `first`: states_host holds `count` payloads of
 * exactly the reference's Vec<i64> encoding, payload i at states_host + i*stride (for PauliNetwork each
 * payload is self-delimiting and `stride` is its allocated slot).  broadcast=1 loads payload 0 into all
 * `count` envs (synth search).  depth := max_depth, internals reset. */
QG_API int qg_set_state(qg_engine* e, const int64_t* states_host, int64_t stride, int64_t first,
                        int64_t count, int32_t broadcast, qg_stream stream);
/* Env::set_state for groups of envs (a search over many targets): payload p (at states_host + p*stride) is loaded into envs
 * [p*group, (p+1)*group) for p < num_states; envs past num_states*group are untouched.  Each payload is packed once on the host.
 * QG_ERR_INVALID for group <= 0 or num_states*group outside the batch. */
QG_API int qg_set_state_grouped(qg_engine* e, const int64_t* states_host, int64_t stride, int64_t num_states, int64_t group,
                                qg_stream stream);
/* Env::reset for every env: identity scrambled by `difficulty` random gates drawn from
 * Philox4x32-10(seed; env id, draw index) (permutation.rs:175-192, linear_function.rs:285-300,
 * clifford.rs:306-319, pauli.rs:554-586).  env ids are first_env_id + local index so a sharded batch
 * draws the same stream as an unsharded one. */
QG_API int qg_reset(qg_engine* e, uint64_t seed, int64_t first_env_id, qg_stream stream);

/* Env::reset restricted to some envs: select_dev uint8[B] (non-zero = reset this env) or NULL = every env whose
 * is_final() holds (depth == 0 or success), which is what a rollout collector does between episodes (twisterl's
 * collectors clone + reset one env per episode; rl/configs.py:133-137 sizes them).  Same Philox streams as qg_reset,
 * so a collector passes a fresh seed per call.  Untouched envs keep their state. */
QG_API int qg_reset_select(qg_engine* e, uint64_t seed, int64_t first_env_id, const uint8_t* select_dev, qg_stream stream);

/* `Clone` of the whole batch (the reference clones one prototype env per episode / rollout,
 * permutation.rs:29, linear_function.rs:154, clifford.rs:179, pauli.rs:307-337): qg_snapshot keeps a
 * device copy of every env record; qg_restore puts it back (solutions restart at the snapshot's length). */
QG_API int qg_snapshot(qg_engine* e, qg_stream stream);
QG_API int qg_restore(qg_engine* e, qg_stream stream);

/* ---- the fused step ------------------------------------------------------------------- */
/* Env::step + reward + is_final + success + observe + masks for all B envs in one launch.
 *  actions_dev  int32[B]            action per env (>= num_actions: state no-op, depth still ticks)
 *  coins_dev    uint8[B] or NULL    injected gen_bool(0.5) results for add_inverts; NULL = Philox
 *  perm_raw_dev uint32[B] or NULL   PauliNetwork+add_perms: raw 32-bit draw for observe()'s perm pick
 *                                   (index = mulhi(raw, n_perms)); NULL = Philox
 *  obs_dev      float[B*obs_size] or NULL   dense 0/1 observation (row-major obs_shape per env)
 *  mask_dev     uint8[B*num_actions] or NULL
 *  reward_dev   float[B] or NULL;  done_dev uint8[B] or NULL (= is_final);  success_dev uint8[B] or NULL */
QG_API int qg_step(qg_engine* e, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev,
                   float* obs_dev, uint8_t* mask_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev,
                   qg_stream stream);
/* `num_steps` consecutive fused steps in ONE launch from a resident action stream: the records are read once, stay
 * in the SM while the steps are played, and are written back once; every step still materialises its observation,
 * mask, reward, done and success exactly as num_steps calls of qg_step would (replaying a solution, evaluating a
 * fixed action stream, the env-throughput benchmark).
 *  actions_dev  int32[num_steps][B];  coins_dev uint8[num_steps][B] or NULL;  perm_raw_dev uint32[num_steps][B] or NULL
 *  obs_dev      float[ring][B][obs_size] or NULL, mask_dev uint8[ring][B][num_actions] or NULL: step t writes slot t % ring
 *  reward_dev   float[num_steps][B] or NULL;  done_dev / success_dev uint8[num_steps][B] or NULL */
QG_API int qg_replay(qg_engine* e, int32_t num_steps, const int32_t* actions_dev, const uint8_t* coins_dev,
                     const uint32_t* perm_raw_dev, float* obs_dev, uint8_t* mask_dev, int32_t ring,
                     float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
/* qg_replay with HOST buffers (pinned recommended): actions_host int32[num_steps][B] (coins_host uint8[num_steps][B] or
 * NULL) go up, reward_host float[num_steps][B] / done_host / success_host uint8[num_steps][B] (each may be NULL) come back;
 * observations / masks stay in the device ring for the policy.  With pinned (page-locked) buffers the whole episode is ONE launch
 * whose kernel reads / writes the host memory itself over PCIe; with pageable buffers chunks of steps are pipelined over a copy-in
 * stream, the caller's stream (one fused launch per chunk) and a copy-out stream (staging buffers allocated on first use).  The call
 * returns when everything has arrived. */
QG_API int qg_replay_host(qg_engine* e, int32_t num_steps, const int32_t* actions_host, const uint8_t* coins_host,
                          float* obs_dev, uint8_t* mask_dev, int32_t ring,
                          float* reward_host, uint8_t* done_host, uint8_t* success_host, qg_stream stream);
/* Same step with HOST buffers (pinned or pageable): actions (and coins) go in, the step runs
 * writing obs/mask to the given DEVICE tensors (may be NULL), reward/done/success come out and the
 * stream is synchronised.  This is the end-to-end call a host-side collector makes.  With pinned
 * (page-locked) buffers the kernel accesses the host memory itself over PCIe (one launch, no
 * staging copies); pageable buffers are staged through device buffers. */
QG_API int qg_step_host(qg_engine* e, const int32_t* actions_host, const uint8_t* coins_host,
                        float* obs_dev, uint8_t* mask_dev,
                        float* reward_host, uint8_t* done_host, uint8_t* success_host, qg_stream stream);

/* ---- stand-alone reads (no state change except the PauliNetwork perm pick) ----------------- */
QG_API int qg_observe(qg_engine* e, const uint32_t* perm_raw_dev, float* obs_dev, qg_stream stream);  /* Env::observe, dense */
QG_API int qg_masks(qg_engine* e, uint8_t* mask_dev, qg_stream stream);                                /* Env::masks */
QG_API int qg_read_status(qg_engine* e, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev,
                          int32_t* depth_dev, qg_stream stream);          /* reward/is_final/success/depth */
QG_API int qg_read_metrics(qg_engine* e, uint32_t* counts_dev /*[B][4]: cnots, cnot layers, layers, gates*/, qg_stream stream);
QG_API int qg_read_errors(qg_engine* e, uint32_t* flags_dev /*[B]*/, qg_stream stream);
/* Raw state of one env in the reference's own byte-per-entry layout (perm: n bytes; LF: n*n;
 * Clifford: 4n*n; PauliNetwork: 2n x (2n+R) row-major, R = rotations loaded), for parity tests. */
QG_API int qg_get_state_host(qg_engine* e, int64_t env, uint8_t* out_host, int64_t cap, int64_t* len, qg_stream stream);
/* Env::solution (solution ++ reverse(solution_inv); PauliNetwork rotation words as pauli.rs:685-719). */
QG_API int qg_solution_host(qg_engine* e, int64_t env, uint32_t* out_host, int32_t cap, int32_t* len, qg_stream stream);

/* Env::solution of MANY envs in one kernel + one copy (clifford.rs:376-381 / pauli.rs:685-719 for `count` envs starting at `first`):
 * row i of out [count][cap] holds the merged action list of env first + i (solution ++ reverse(solution_inv); PauliNetwork words as logged),
 * len[i] its length; a solution longer than `cap` sets len[i] = -(length) and writes nothing.  The _dev form is asynchronous on the stream and
 * writes device buffers; the _host form stages through engine-owned device buffers (grown on first use) and synchronises. */
QG_API int qg_solutions(qg_engine* e, int64_t first, int64_t count, uint32_t* out_dev, int32_t cap, int32_t* len_dev, qg_stream stream);
QG_API int qg_solutions_host(qg_engine* e, int64_t first, int64_t count, uint32_t* out_host, int32_t cap, int32_t* len_host, qg_stream stream);

/* ---- packed host wire format -------------------------------------------------------------------------------------------------
 * qg_replay_host with the narrowest streams the data allows (the host link is what bounds a multi-GPU node end to end):
 *  actions8_host  uint8[num_steps][B]      one byte per action (needs num_actions <= 256; a value >= num_actions is the reference's no-op)
 *  reward_host    float[num_steps][B] or NULL (NULL: rewards stay on the device: pass reward_dev to keep them for a device-side return / qg_gae)
 *  reward_dev     float[num_steps][B] or NULL
 *  done_bits_host, success_bits_host  uint32[ceil(B/32)][num_steps] (success may be NULL): bit (env % 32) of word [env / 32][t] = is_final /
 *                 success of env after step t: 2 bits per env-step, each tile's 32 consecutive steps written as one 128-byte line
 * Buffers must be pinned (qg_host_alloc, cudaHostAlloc, cudaHostRegister): the kernel writes the outputs over PCIe itself and reads the inputs
 * either the same way (small episodes) or from a device staging buffer that the copy engine fills in chunks while the kernel runs (>= 1 MB of
 * actions); one launch per episode; QG_ERR_INVALID for pageable memory.  Observations / masks go to the device ring as in qg_replay. */
QG_API int qg_replay_host_packed(qg_engine* e, int32_t num_steps, const uint8_t* actions8_host, const uint8_t* coins_host,
                                 float* obs_dev, uint8_t* mask_dev, int32_t ring, float* reward_host, float* reward_dev,
                                 uint32_t* done_bits_host, uint32_t* success_bits_host, qg_stream stream);
/* The same call without the final synchronisation: returns once everything is queued on `stream`; the host buffers are the call's until the
 * stream (or an event recorded on it after the call) has been waited for.  A collector keeps two episodes in flight — queue episode k + 1 (its
 * own output buffers), then wait for episode k and read its rewards / flags — so the device never idles across the host's turn-around.
 * Neither form can be captured into a CUDA graph (the staged inputs use a second, engine-owned stream). */
QG_API int qg_replay_host_packed_async(qg_engine* e, int32_t num_steps, const uint8_t* actions8_host, const uint8_t* coins_host,
                                       float* obs_dev, uint8_t* mask_dev, int32_t ring, float* reward_host, float* reward_dev,
                                       uint32_t* done_bits_host, uint32_t* success_bits_host, qg_stream stream);
/* The device-resident form of the same formats (actions8_dev uint8[num_steps][B], bit planes on the device). */
QG_API int qg_replay_packed(qg_engine* e, int32_t num_steps, const uint8_t* actions8_dev, const uint8_t* coins_dev,
                            float* obs_dev, uint8_t* mask_dev, int32_t ring, float* reward_dev,
                            uint32_t* done_bits_dev, uint32_t* success_bits_dev, qg_stream stream);
/* Pinned host memory on the NUMA node the GPU hangs off (sysfs numa_node of its PCI function): the calling thread is bound to that node's
 * CPUs and its memory policy to that node while the pages are allocated and first touched, then both are restored.  On a multi-GPU host
 * this keeps every GPU's PCIe traffic on its own socket's memory controllers.  Falls back to plain cudaHostAlloc where the topology cannot
 * be read.  *numa_node_out (may be NULL) receives the node used, -1 if unknown. */
QG_API int qg_host_alloc(int32_t device, size_t bytes, void** out_host, int32_t* numa_node_out);
QG_API int qg_host_free(void* host);
/* Binds the calling host thread to the CPUs of the GPU's NUMA node (the thread that drives an engine should run there). Returns the node or -1. */
QG_API int qg_bind_thread_to_device(int32_t device);

/* ---- zero-copy observations for the policy (DLPack) ----------------------------------------------------------------------------
 * The engine allocates (once) an observation ring float[ring][B][rows][cols] and hands it out as a DLManagedTensor* (DLPack v0.8 ABI, device
 * kDLCUDA, dtype float32; shape (B, rows, cols) for ring == 1): wrap it in a PyCapsule named "dltensor" for torch.from_dlpack, or consume it
 * from Rust / C++ directly.  *obs_dev_out receives the same pointer for qg_step / qg_replay's obs_dev argument.  The memory belongs to the
 * engine (freed by qg_destroy): the tensor must not outlive it; the deleter only frees the descriptor. */
QG_API int qg_dlpack_obs(qg_engine* e, int32_t ring, void** managed_tensor_out, float** obs_dev_out);

/* ---- synth search (rollout driver pieces around the policy) ---------------------------- */
/* Starts a search over the engine's B rollouts: zeroes the per-rollout return accumulators.
 * The caller loads the target first (qg_set_state broadcast=1). */
QG_API int qg_search_begin(qg_engine* e, uint64_t seed, int64_t first_rollout_id, qg_stream stream);
/* One decision for every rollout that is not final yet: pick an action from the policy's
 * non-negative action weights (weights_dev float[B*num_actions], e.g. softmax probabilities; masked by
 * Env::masks), deterministic=1: first arg-max; 0: inverse-CDF sample with a Philox uniform and a
 * sequential f32 cumulative sum; then the fused step; return += reward.  Final rollouts are left
 * untouched.  chosen_dev int32[B] or NULL receives the action (-1 for rollouts already final). */
QG_API int qg_search_step(qg_engine* e, const float* weights_dev, int32_t deterministic,
                          float* obs_dev, uint8_t* mask_dev, int32_t* chosen_dev, int32_t* num_active_dev, qg_stream stream);
/* On-GPU best-rollout reduction: key = success<<62 | orderable(return)<<30 | (2^30-1 - rollout id)
 * (max wins: successful first, then highest return, then lowest id).  Writes the winning key to
 * *best_key_host and the winner's local env index to *best_env_host (-1 if B == 0). */
QG_API int qg_search_best(qg_engine* e, int64_t* best_key_host, int64_t* best_env_host, qg_stream stream);
/* Per-target best rollout of a search over many targets (each target loaded into its own group of rollouts by qg_set_state_grouped):
 * for every group g of envs [g*group, (g+1)*group), g < num_groups, keys_dev[g] = the largest qg_search_best key of the group, and if
 * that rollout succeeded, actions_dev[g][0..len) its Env::solution with len_dev[g] = len (len_dev[g] = 0: no rollout of the group
 * succeeded; -(length): the solution is longer than cap and nothing is written).  keys_dev int64[num_groups], actions_dev
 * uint32[num_groups][cap], len_dev int32[num_groups].  One kernel, asynchronous on the stream, no host synchronisation. */
QG_API int qg_search_best_grouped(qg_engine* e, int64_t group, int64_t num_groups, int64_t* keys_dev, uint32_t* actions_dev, int32_t cap,
                                  int32_t* len_dev, qg_stream stream);
QG_API int qg_read_returns(qg_engine* e, float* returns_dev, qg_stream stream);
/* End of a search sharded over GPUs (rl/synthesis.py:112-126 `solve(..., num_searches)` with the rollouts split over ranks, each rank's
 * qg_search_begin given its first GLOBAL rollout id): the on-GPU best-rollout reduction of this rank, then — given an NCCL communicator —
 * ONE all-gather of every rank's (key, solution length, action list) row and an on-GPU pick of the largest key, so that every rank ends with
 * the same winner without a host decision in between.  comm: an ncclComm_t (qg_nccl_comm_create below, or any communicator of the same NCCL
 * library whose ranks all make this call), or NULL for a single GPU.  Outputs (host): *best_key_host the winning packed key (0: no rollout),
 * *success_host, *rollout_id_host its global rollout id, *owner_rank_host, actions_host[0..*len_host) the winner's Env::solution (only when
 * it succeeded and fits `cap`; *len_host = 0 otherwise).  Identical results for any number of ranks (keys embed the global rollout id). */
typedef struct ncclComm* qg_nccl_comm;
QG_API int qg_search_finish(qg_engine* e, qg_nccl_comm comm, int64_t* best_key_host, int32_t* success_host, int64_t* rollout_id_host,
                            int32_t* owner_rank_host, uint32_t* actions_host, int32_t cap, int32_t* len_host, qg_stream stream);
/* NCCL plumbing for hosts without torch (the library is loaded with dlopen("libnccl.so.2") on first use; QG_ERR_UNSUPPORTED if absent):
 * rank 0 makes an id and ships the 128 bytes to the others by any channel; every rank then creates its communicator on its device. */
QG_API int qg_nccl_unique_id(uint8_t id_out[128]);
QG_API int qg_nccl_comm_create(const uint8_t id[128], int32_t rank, int32_t world, int32_t device, qg_nccl_comm* out);
QG_API int qg_nccl_comm_destroy(qg_nccl_comm comm);

/* ---- rollout collector pieces (the data-collection half of twisterl's PPO loop, SURVEY.md §8f row 1) ------------- */
/* qg_search_step that also reports the step's reward / is_final / success per env (entries of envs that were already
 * final, chosen = -1, are left untouched) and takes the Philox seed of this decision explicitly: the action sample of
 * env i is drawn from (seed; first_env_id + i, env's step counter, sample stream). */
QG_API int qg_collect_step(qg_engine* e, uint64_t seed, const float* weights_dev, int32_t deterministic,
                           float* obs_dev, uint8_t* mask_dev, int32_t* chosen_dev,
                           float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
/* The two collector calls with the Philox seed of the decision read from DEVICE memory when the kernel runs (*seed_dev), so that a decision —
 * or a whole rollout of decisions — captured in a CUDA graph can be replayed with fresh seeds: the host rewrites the seed words between
 * replays.  Otherwise identical to qg_reset_select / qg_collect_step. */
QG_API int qg_reset_select_dev(qg_engine* e, const uint64_t* seed_dev, int64_t first_env_id, const uint8_t* select_dev, qg_stream stream);
QG_API int qg_collect_step_dev(qg_engine* e, const uint64_t* seed_dev, const float* weights_dev, int32_t deterministic,
                               float* obs_dev, uint8_t* mask_dev, int32_t* chosen_dev,
                               float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
/* qg_collect_step_dev for a collector with twists: weights_dev float[B][A] are in the policy's (twisted) action order and env action g of
 * env i takes the weight weights[i][act_perm[twist[i]][g]] (act_perm_dev int32[K][A], the act_perms of qg_twists_copy; twist_dev int32[B]).
 * The pick is bit-identical to qg_twist_gather(weights, act_perm, twist) followed by qg_collect_step_dev, without the gathered copy.
 * policy_chosen_dev (int32[B], may be NULL): the chosen action in the policy's order, act_perm[twist[i]][chosen], or -1 where chosen is -1.
 * No observation / mask output. */
QG_API int qg_collect_step_twisted_dev(qg_engine* e, const uint64_t* seed_dev, const float* weights_dev, const int32_t* act_perm_dev,
                                       const int32_t* twist_dev, int32_t deterministic, int32_t* chosen_dev, int32_t* policy_chosen_dev,
                                       float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
/* Generalised advantage estimation over a rollout laid out [num_steps][batch] (value_dev has num_steps + 1 rows, the
 * last one bootstraps the truncated episodes):  nd = !done[t];  delta = (reward[t] + (gamma*value[t+1])*nd) - value[t];
 * adv[t] = delta + ((gamma*lambda)*nd)*adv[t+1];  ret[t] = adv[t] + value[t]  — f32, every operation rounded on its
 * own in that order.  valid_dev (uint8, may be NULL): 0 marks a slot where the env was not stepped (adv = ret = 0).
 * Needs no engine: plain device pointers. */
QG_API int qg_gae(const float* reward_dev, const float* value_dev, const uint8_t* done_dev, const uint8_t* valid_dev,
                  int32_t num_steps, int64_t batch, float gamma, float lambda, float* adv_dev, float* ret_dev, qg_stream stream);
/* Twists on the device (Env::twists, symmetry.rs:297-361): out[b][j] = in[b][table[index[b]][j]] for an int32 table
 * [K][len] and a per-env twist index int32[B] (NULL = twist 0).  With the inverse of obs_perms[k] this is the twisted
 * observation (entry i moves to obs_perms[k][i]); with act_perms[k] it brings the policy's action weights back into
 * the env's action order. */
QG_API int qg_twist_gather(const float* in_dev, float* out_dev, const int32_t* table_dev, const int32_t* index_dev,
                           int64_t batch, int32_t len, qg_stream stream);
/* Twists on packed observations (Permutation / LinearFunction / Clifford: every obs perm is the lift of a qubit permutation p, entry (r, c) of
 * the dim x dim observation -> (lift(r), lift(c)), lift(i) = p[i] for i < n, n + p[i - n] otherwise; dim = n or 2n).  qperm_inv_dev uint8
 * [num_twists][num_qubits] holds p^-1 per twist; out_bits = the packed bits of qg_twist_gather(unpacked in_bits, inverse obs perm, k).  The
 * twist index k of env b is index_dev[b] when given, else drawn on the device: mulhi(philox(*seed_dev; first_env_id + b, draw, stream 5),
 * num_twists), and written to index_out_dev[b] when that is not NULL.  in_bits / out_bits uint32[batch][ceil(obs_size / 32)], not in place. */
QG_API int qg_twist_bits(const uint32_t* in_bits_dev, uint32_t* out_bits_dev, int64_t batch, int32_t obs_size, int32_t num_qubits, int32_t dim,
                         const uint8_t* qperm_inv_dev, int32_t num_twists, const int32_t* index_dev, const uint64_t* seed_dev,
                         int64_t first_env_id, int32_t draw, int32_t* index_out_dev, qg_stream stream);

/* ---- packed-bit observations + fused policy network (SURVEY.md §8f row 3) ------------------------------------------
 * Env::observe returns the indices of the non-zero entries (e.g. clifford.rs:361-368) because twisterl's policy sums
 * first-layer weight columns over them.  The *_bits entry points deliver the same information as one bit per entry:
 * obs_bits_dev uint32[B][qg_obs_words] (bit i%32 of word i/32 = entry i of the row-major observation), 32x smaller
 * than the dense f32 tensor; everything else is identical to the entry point of the same name without the suffix. */
typedef struct qg_policy qg_policy;
QG_API int32_t qg_obs_words(const qg_engine* e);            /* ceil(obs_size / 32) */
QG_API int qg_step_bits(qg_engine* e, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev,
                        uint32_t* obs_bits_dev, uint8_t* mask_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev,
                        qg_stream stream);
QG_API int qg_replay_bits(qg_engine* e, int32_t num_steps, const int32_t* actions_dev, const uint8_t* coins_dev,
                          const uint32_t* perm_raw_dev, uint32_t* obs_bits_dev, uint8_t* mask_dev, int32_t ring,
                          float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
QG_API int qg_observe_bits(qg_engine* e, const uint32_t* perm_raw_dev, uint32_t* obs_bits_dev, qg_stream stream);
QG_API int qg_search_step_bits(qg_engine* e, const float* weights_dev, int32_t deterministic, uint32_t* obs_bits_dev,
                               int32_t* chosen_dev, int32_t* num_active_dev, qg_stream stream);
/* The action network of a twisterl BasicPolicy (the .pt files under examples/models: embeddings -> ReLU -> common[i] -> ReLU ... ->
 * action head) evaluated from packed observations in one kernel: first layer = bias + sum of the weight columns of the
 * set bits, then the Linear/ReLU chain and a softmax.  Layer l has out_features[l] outputs and consumes the
 * observation (l = 0) or layer l-1; weights_host[l] is torch's Linear.weight layout [out][in] row-major, f32; ReLU
 * follows every layer but the last.  Limits: 1..8 layers, widths <= 1024 (the last layer's width counts the value column of
 * qg_policy_create_value), and the CTA's shared-memory plan must fit 210 KB, which caps obs_size well below 65535 (QG_ERR_UNSUPPORTED).
 * Arithmetic (tests/test_policy_fused_envelope.py restates it bit for bit):
 * - First layer: its input is 0/1, so it is a sum of weight rows, computed EXACTLY.  The weights (with the value column when the network
 *   has one layer) are converted once to fixed point, q = rint(w * 2^shift) with ties to even, shift = min(30 - e, 120) where
 *   2^(e-1) <= max |w| < 2^e (shift = 30 when every weight is 0), and summed in 64-bit integers; then h = b + float(float(sum) * 2^-shift)
 *   in f32.  The sum is independent of the order of its terms, which lets qg_search_run update it from the observation entries that
 *   changed instead of recomputing it, with bit-identical results.
 * - Other layers: f32 fused multiply-adds in partial chains over the inputs, combined with f32 adds in a fixed order.  The inputs are
 *   read in tiles of kt = max(1, 8192 / stride) rows, stride = the layer's width rounded up to a multiple of 4, and split by their
 *   position u within the tile (not by their global index):
 *     width > 256:      2 chains, chain c takes u = c, c + 2, ..;  chain 0 starts from the bias, chain 1 from 0;  z = c0 + c1
 *     width 65..256:    4 chains, u = c, c + 4, ..;  chain 0 starts from the bias, the others from 0;  z = ((c0 + c1) + c2) + c3
 *     width <= 64:      16 chains, u = c, c + 16, .., all start from 0;  z = ((((0 + c0) + c1) + ..) + c15) + b
 *   Each chain runs over the tiles in order.  The order is fixed by the shape alone, so a row's outputs do not depend on the batch,
 *   the other rows or the launch, and qg_search_run decides exactly as the per-decision launches do.
 * - Softmax over the A action logits (the value column is not part of it): lane l of a warp takes a = l, l + 32, .. for the max and
 *   the sum of expf(z - max), the lanes are combined by an xor butterfly (offsets 16, 8, 4, 2, 1), p = expf(z - max) * (1 / sum). */
QG_API int qg_policy_create(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features,
                            const float* const* weights_host, const float* const* biases_host, qg_policy** out);
/* The same with the BasicPolicy's value head (a single Linear from the last common layer to one output, examples/models/{*}.pt
 * `value.0.weight [1][in]`, `value.0.bias`): it is evaluated as one more output of the last layer, outside the softmax, and read with
 * qg_policy_forward_bits_value.  value_weight_host: float[in_features of the last layer], or NULL for no value head. */
QG_API int qg_policy_create_value(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features,
                                  const float* const* weights_host, const float* const* biases_host,
                                  const float* value_weight_host, float value_bias, qg_policy** out);
QG_API void qg_policy_destroy(qg_policy* p);
QG_API int32_t qg_policy_num_actions(const qg_policy* p);
QG_API int32_t qg_policy_has_value(const qg_policy* p);
/* probs_dev float[B][num_actions] (softmax) and / or logits_dev float[B][num_actions]; either may be NULL. */
QG_API int qg_policy_forward_bits(qg_policy* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev,
                                  float* logits_dev, qg_stream stream);
/* ... and values_dev float[B] (the value head's output; the policy must have been created with one); any of the three may be NULL. */
QG_API int qg_policy_forward_bits_value(qg_policy* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev,
                                        float* logits_dev, float* values_dev, qg_stream stream);

/* The same network for LARGE batches (the rollout collector: tens of thousands of envs per decision) on the 5th-generation tensor cores
 * (csrc/qg_policy_tc.cu: tcgen05.mma with tensor-memory accumulators, bulk-copy operand pipeline).  Every f32 value travels as two f16
 * halves (hi + lo, 22 significant bits) and every product as hi*hi + hi*lo + lo*hi with f32 accumulation, so logits stay within the f32
 * module's 1e-4 tolerance.  Arguments as qg_policy_create_value; max_batch sizes the activation buffers (allocated once, here); at most
 * 127 actions; sm_100 only (QG_ERR_UNSUPPORTED elsewhere).  forward: probs / logits float[B][num_actions], values float[B] (any may be NULL). */
typedef struct qg_policy_tc qg_policy_tc;
QG_API int qg_policy_tc_create(int32_t device, int32_t obs_size, int32_t num_layers, const int32_t* out_features,
                               const float* const* weights_host, const float* const* biases_host,
                               const float* value_weight_host, float value_bias, int64_t max_batch, qg_policy_tc** out);
QG_API void qg_policy_tc_destroy(qg_policy_tc* p);
QG_API int32_t qg_policy_tc_num_actions(const qg_policy_tc* p);
/* A three-layer policy whose padded widths fit (embeddings a multiple of 128, common layer <= 256) runs as ONE kernel that keeps the hidden
 * activations on chip; per_layer = 1 forces the one-kernel-per-layer path instead (same arithmetic).  Returns 1 if the fused kernel will run. */
QG_API int32_t qg_policy_tc_set_mode(qg_policy_tc* p, int32_t per_layer);
QG_API int qg_policy_tc_forward_bits(qg_policy_tc* p, const uint32_t* obs_bits_dev, int64_t batch, float* probs_dev, float* logits_dev,
                                     float* values_dev, qg_stream stream);
/* Refreshes the handle's weights in place from f32 DEVICE tensors (a training loop's parameters): the same hi / lo split as
 * qg_policy_tc_create, stream-ordered, no allocation, every device pointer kept — a CUDA graph captured with this handle stays valid.  The
 * shapes (obs_size, num_layers, out_features, value head present or not) must equal those of creation.  weights_dev[l] float[out][in]
 * row-major, biases_dev[l] float[out], value_weight_dev float[in of the last layer], value_bias_dev float[1] (both NULL without a value head). */
QG_API int qg_policy_tc_load_weights_dev(qg_policy_tc* p, int32_t obs_size, int32_t num_layers, const int32_t* out_features,
                                         const float* const* weights_dev, const float* const* biases_dev,
                                         const float* value_weight_dev, const float* value_bias_dev, qg_stream stream);
/* Training on the tensor cores.  enable_training allocates, once, what the backward pass needs for up to max_batch rows (dZ images of every
 * layer, transposed weight images, split-K partials); later weight loads keep them current.  generation() counts forwards.  backward
 * differentiates the handle's latest forward, which must have run one kernel per layer (qg_policy_tc_set_mode(p, 1)) with `batch` rows and
 * have been generation `generation` (QG_ERR_INVALID otherwise): dlogits_dev float[batch][num_actions], dvalues_dev float[batch] (NULL = 0)
 * -> grad_w_dev[l] float[out][in], grad_b_dev[l] float[out], grad_vw_dev float[in of the last layer], grad_vb_dev float[1], OVERWRITTEN.
 * Same split-f16 arithmetic as the forward; the head's gradient is scaled by a power of two chosen on the device; weight gradients are
 * summed over 1024-row chunks and the chunks in a fixed order, so they are bit-reproducible.  Stream-ordered, allocates nothing. */
QG_API int qg_policy_tc_enable_training(qg_policy_tc* p);
QG_API int64_t qg_policy_tc_generation(const qg_policy_tc* p);
QG_API int qg_policy_tc_backward(qg_policy_tc* p, int64_t generation, int64_t batch, const float* dlogits_dev, const float* dvalues_dev,
                                 float* const* grad_w_dev, float* const* grad_b_dev, float* grad_vw_dev, float* grad_vb_dev, qg_stream stream);

/* The whole rollout search in ONE launch: every CTA owns 8 rollouts and loops  policy (packed observation -> action weights) ->
 * sample / arg-max + fused step -> next packed observation  until its rollouts are final or max_decisions decisions were taken;
 * equivalent to max_decisions rounds of qg_policy_forward_bits + qg_search_step_bits (same bits), without launch gaps or host
 * round trips.  Call qg_set_state (broadcast), qg_search_begin and qg_observe_bits first; obs_bits_dev uint32[B][qg_obs_words]
 * holds the initial packed observations (read only: during the search the records, the returns and the observation bits stay on chip
 * and only the final records / returns are written back), weights_dev float[B][num_actions] is reserved; decisions_dev
 * int32[ceil(B/8)] (or NULL) receives the number of decisions each CTA took.  Then qg_search_best / qg_solution_host as usual.
 * Grows a per-policy scratch buffer (8 x width[0] int64 per CTA) on first use with a larger batch: one host thread per policy handle. */
QG_API int qg_search_run(qg_engine* e, qg_policy* policy, int32_t deterministic, int32_t max_decisions, uint32_t* obs_bits_dev,
                         float* weights_dev, int32_t* decisions_dev, qg_stream stream);

/* The twisted rollout search: the policy runs in a symmetry frame of the env (its twists, qg_twists_copy of a config with add_perms = 1)
 * drawn per rollout and decision, as the collector trains it.  Protocol: rollout i (global id g = first_rollout_id + i of qg_search_begin)
 * decides in frame k = mulhi(philox(seed; g, tick, stream 5), num_twists), tick = its step counter at decision time (the counter that
 * also keys the decision's sample draw), so k depends on the seed, g and the decision index only.  The policy sees the observation in
 * frame k (entry i moves to obs_perms[k][i], as qg_twist_bits); env action a weighs probs[act_perm[k][a]] and the arg-max / inverse-CDF
 * sum run over a in env order (as qg_collect_step_twisted_dev).  Returns, solutions (env action order), keys and the best-rollout rule are
 * those of the untwisted search; a table holding only the identity reproduces it bit for bit.
 * Tables (device memory, the caller's): qperm_inv_dev uint8[num_twists][num_qubits], the inverse qubit permutation of every twist (as for
 * qg_twist_bits); act_perm_dev int32[num_twists][num_actions], the act perms; twist_dev int32[B], each rollout's frame of its current
 * decision (written by these calls).  Permutation (<= 64 qubits), LinearFunction and Clifford; QG_ERR_UNSUPPORTED for PauliNetwork (its
 * symmetry is applied inside the env by add_perms) and for a Permutation without packed observations.
 * - qg_search_observe_twisted: after qg_set_state and qg_search_begin, the packed observations of the rollouts in the frame of their next
 *   decision (drawn from their step counters) -> obs_bits_dev uint32[B][qg_obs_words], the frames -> twist_dev.
 * - qg_search_step_twisted: the counterpart of qg_search_step_bits: picks through act_perm[twist[i]], steps, and writes the next
 *   observation already in the frame drawn from the post-step tick, updating twist_dev.
 * - qg_search_run_twisted: qg_search_run for the twisted search, obs_bits_dev / twist_dev as qg_search_observe_twisted left them; its
 *   decisions are bit-identical to rounds of qg_policy_forward_bits + qg_search_step_twisted. */
QG_API int qg_search_observe_twisted(qg_engine* e, uint32_t* obs_bits_dev, const uint8_t* qperm_inv_dev, int32_t num_twists, int32_t* twist_dev,
                                     qg_stream stream);
QG_API int qg_search_step_twisted(qg_engine* e, const float* weights_dev, int32_t deterministic, uint32_t* obs_bits_dev,
                                  const uint8_t* qperm_inv_dev, const int32_t* act_perm_dev, int32_t num_twists, int32_t* twist_dev,
                                  int32_t* chosen_dev, int32_t* num_active_dev, qg_stream stream);
QG_API int qg_search_run_twisted(qg_engine* e, qg_policy* policy, int32_t deterministic, int32_t max_decisions, uint32_t* obs_bits_dev,
                                 float* weights_dev, int32_t* decisions_dev, const uint8_t* qperm_inv_dev, const int32_t* act_perm_dev,
                                 int32_t num_twists, int32_t* twist_dev, qg_stream stream);

/* ---- tree search (SURVEY.md §8f row 4: num_mcts_searches > 0, rl/synthesis.py:122-124, rl/configs.py:30-42) ----------------
 * Clone + step through record slots: the engine's batch is a pool of record slots; logical env i (i < count) reads the
 * record in slot src_slot_dev[i], plays actions_dev[i] and writes the result to slot dst_slot_dev[i] (a tree-search child
 * node = clone of the parent's env + one step, the reference's `Clone` + `step`).  A negative action leaves slot and outputs
 * of env i untouched.  Outputs (each may be NULL) are indexed by i like qg_step's. */
QG_API int qg_step_slots(qg_engine* e, int64_t count, const int32_t* src_slot_dev, const int32_t* dst_slot_dev,
                         const int32_t* actions_dev, float* obs_dev, uint32_t* obs_bits_dev, uint8_t* mask_dev,
                         float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream);
/* Copies the records of envs 0..count-1 of `src` into the slots dst_slot_dev[i] of `dst` (same env kind, qubits and gateset;
 * batch and track_solution may differ: the copies restart their solution log). */
QG_API int qg_copy_records(qg_engine* dst, const int32_t* dst_slot_dev, qg_engine* src, int64_t count, qg_stream stream);

/* Device arrays of num_trees PUCT trees with node_cap nodes each (caller-owned, see csrc/qg_mcts.cu for the protocol);
 * node j of tree i lives in record slot i * node_cap + j of the slot-pool engine. */
typedef struct qg_mcts_tree {
    int32_t num_trees, node_cap, num_actions;
    float* prior;          /* [num_trees][node_cap][num_actions] */
    int32_t* visits;       /* [num_trees][node_cap][num_actions] */
    float* value_sum;      /* [num_trees][node_cap][num_actions] */
    int32_t* child;        /* [num_trees][node_cap][num_actions] node index or -1 */
    float* node_reward;    /* [num_trees][node_cap] reward of the step that created the node */
    uint8_t* node_final;   /* [num_trees][node_cap] */
    int32_t* node_count;   /* [num_trees] */
    int32_t* path_node;    /* [num_trees][node_cap] */
    int32_t* path_action;  /* [num_trees][node_cap] */
    int32_t* path_len;     /* [num_trees] */
    int32_t* new_node;     /* [num_trees] node created by the last select, -1 if none */
} qg_mcts_tree;
/* New decision: node 0 of every tree gets root_prior_dev float[num_trees][num_actions] and root_final_dev uint8[num_trees]. */
QG_API int qg_mcts_begin(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, qg_stream stream);
/* One simulation's descent per tree; writes the slots / action of the expansion for qg_step_slots (action -1: none). */
QG_API int qg_mcts_select(const qg_mcts_tree* t, float c_puct, int32_t* src_slot_dev, int32_t* dst_slot_dev,
                          int32_t* action_dev, qg_stream stream);
/* Finishes the simulation: the new node gets prior_dev float[num_trees][num_actions], reward_dev / done_dev of its step and
 * value_dev float[num_trees] (ignored if final); returns are backed up along the recorded path. */
QG_API int qg_mcts_backup(const qg_mcts_tree* t, const float* prior_dev, const float* value_dev, const float* reward_dev,
                          const uint8_t* done_dev, qg_stream stream);
/* weights_dev float[num_trees][num_actions] = root visit counts / their sum (all zero for a tree without simulations). */
QG_API int qg_mcts_root_weights(const qg_mcts_tree* t, float* weights_dev, qg_stream stream);
/* Tree reuse between decisions (protocol in csrc/qg_mcts.cu), after the rollouts' qg_search_step with chosen_dev int32[num_trees]: tree i
 * is re-rooted at c = child[0][chosen[i]] when chosen[i] >= 0, that child exists and its record in `pool` (slot i * node_cap + c) equals env
 * i's record in `rollouts` (solution-log length masked).  It then keeps the first keep_nodes (1..node_cap) nodes of c's subtree in creation
 * order, renumbered in that order (c becomes node 0), with their pool records; an edge whose child was dropped keeps N / W and gets child
 * -1.  reused_dev uint8[num_trees] receives 1 for a re-rooted tree, 0 otherwise (the tree is left for qg_mcts_begin_keep to start
 * afresh).  Uses path_node as scratch (it is free between decisions).  `pool` and `rollouts` share env kind, qubits, gateset and device. */
QG_API int qg_mcts_reroot(const qg_mcts_tree* t, qg_engine* pool, const qg_engine* rollouts, const int32_t* chosen_dev, int32_t keep_nodes,
                          uint8_t* reused_dev, qg_stream stream);
/* qg_mcts_begin for the trees with reused_dev[i] == 0; re-rooted trees (reused_dev[i] != 0) are left untouched, root prior included. */
QG_API int qg_mcts_begin_keep(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, const uint8_t* reused_dev,
                              qg_stream stream);

/* The twisted tree search: every policy evaluation of a tree runs in a symmetry frame of the env (its twists, qg_twists_copy of a config
 * with add_perms = 1).  Tree i belongs to the rollout with global id g = first_rollout_id + i; evaluation e = 0 is its root, e = s + 1 the
 * leaf created by simulation s of the decision.  Its frame is  k(i, e) = mulhi(philox(seed; g + (e << 32), tick_i, stream 5), num_twists),
 * tick_i = the rollout's step counter at decision time, so k(i, 0) is the frame qg_search_observe_twisted draws.  The policy sees the node's
 * observation in frame k (entry j moves to obs_perms[k][j], as qg_twist_bits); the node stores its prior in env action order,
 * P(a) = probs[act_perm[k][a]]; the value is used as is.  PUCT, back-up, root weights, re-rooting and the decision do not change.  A table
 * holding only the identity reproduces the untwisted search bit for bit.  Permutation (<= 64 qubits), LinearFunction and Clifford;
 * QG_ERR_UNSUPPORTED for PauliNetwork and for a Permutation without packed observations.
 * search_key_dev uint64[2] = {seed, first_rollout_id} (those of qg_search_begin) and eval_dev int32[1] = the current evaluation index minus
 * one are read in device memory when the kernels run, so one captured CUDA graph serves every decision and every seed: the caller rewrites
 * search_key_dev when the search restarts.  Tables: qperm_inv_dev uint8[num_twists][num_qubits] and act_perm_dev int32[num_twists][num_actions]
 * as for qg_search_run_twisted; twist_dev int32[num_trees] holds the frame of each tree's last evaluation.
 * - qg_mcts_observe_twisted, root pass (pool NULL): the root observations, read from `rollouts` records, in frames k(i, 0) ->
 *   obs_bits_dev uint32[num_trees][qg_obs_words], the frames -> twist_dev; resets *eval_dev to 0.  Leaf pass (after qg_mcts_select and
 *   qg_step_slots): tree i with action_dev[i] >= 0 observes pool slot dst_slot_dev[i] in frame k(i, *eval_dev + 1); the other trees' rows
 *   and frames are left untouched.  The tick and the ids come from `rollouts`, which must not step during the decision.
 * - qg_mcts_begin_twisted / qg_mcts_begin_keep_twisted: qg_mcts_begin / qg_mcts_begin_keep with root_prior_dev in frames twist_dev.
 * - qg_mcts_backup_twisted: qg_mcts_backup with prior_dev in frames twist_dev; then advances *eval_dev by one (the simulation is over). */
QG_API int qg_mcts_observe_twisted(const qg_engine* rollouts, const qg_engine* pool, const int32_t* dst_slot_dev, const int32_t* action_dev,
                                   const uint64_t* search_key_dev, int32_t* eval_dev, const uint8_t* qperm_inv_dev, int32_t num_twists,
                                   uint32_t* obs_bits_dev, int32_t* twist_dev, qg_stream stream);
QG_API int qg_mcts_begin_twisted(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, const int32_t* act_perm_dev,
                                 int32_t num_twists, const int32_t* twist_dev, qg_stream stream);
QG_API int qg_mcts_begin_keep_twisted(const qg_mcts_tree* t, const float* root_prior_dev, const uint8_t* root_final_dev, const uint8_t* reused_dev,
                                      const int32_t* act_perm_dev, int32_t num_twists, const int32_t* twist_dev, qg_stream stream);
QG_API int qg_mcts_backup_twisted(const qg_mcts_tree* t, const float* prior_dev, const float* value_dev, const float* reward_dev,
                                  const uint8_t* done_dev, const int32_t* act_perm_dev, int32_t num_twists, const int32_t* twist_dev,
                                  int32_t* eval_dev, qg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* QG_ENGINE_H */
