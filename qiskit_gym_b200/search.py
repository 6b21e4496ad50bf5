"""Synth-time rollout search on the device (the `num_searches` policy-guided rollouts of
`RLSynthesis.synth`, reference src/qiskit_gym/rl/synthesis.py:112-126 -> twisterl `Algorithm.solve`).

Per decision step, for all rollouts at once:   observation (device tensor, written by the previous fused step)
-> PyTorch policy MLP -> softmax -> `qg_search_step` (masked arg-max / Philox sampling + fused env step +
return accumulation + action log).  One iteration is captured in a CUDA graph and replayed; the best rollout is
reduced on the GPU (`qg_search_best`) and, across ranks, with one int64 MAX all-reduce plus a broadcast of the
winning action list.

twisterl is not in the reference tree, so its exact rollout protocol is *unpinned* (SURVEY.md §8c): what is
fixed here is  (a) final rollouts stop stepping, (b) best = (success, sum of rewards, lowest rollout id),
(c) `None` when no rollout succeeds (rl/synthesis.py:125).
"""
from __future__ import annotations

import time
from dataclasses import dataclass

import numpy as np
import torch

from . import _abi
from .engine import BatchedEnv

KEY_SUCCESS_BIT = 62
KEY_ID_MASK = 0x3FFFFFFF


class BasicPolicy(torch.nn.Module):
    """MLP with the parameter names/shapes of twisterl's `BasicPolicy` as saved in the reference's
    examples/models/*.pt: embeddings.{weight[E,obs],bias}, common.{i}.{weight,bias}, action.0.*, value.0.*.
    (Activation placement is recalled, not verifiable here: ReLU after the embedding and after each common layer.)"""

    def __init__(self, obs_shape, num_actions, embedding_size=512, common_layers=(256,), policy_layers=(), value_layers=()):
        super().__init__()
        obs = 1
        for d in obs_shape:
            obs *= int(d)
        self.embeddings = torch.nn.Linear(obs, embedding_size)
        layers, last = [], embedding_size
        for h in common_layers:
            layers += [torch.nn.Linear(last, h), torch.nn.ReLU()]
            last = h
        self.common = torch.nn.Sequential(*layers)

        def head(hidden, out):
            ls, l = [], last
            for h in hidden:
                ls += [torch.nn.Linear(l, h), torch.nn.ReLU()]
                l = h
            ls.append(torch.nn.Linear(l, out))
            return torch.nn.Sequential(*ls)

        self.action = head(tuple(policy_layers), num_actions)
        self.value = head(tuple(value_layers), 1)

    def forward(self, obs):
        x = torch.relu(self.embeddings(obs.reshape(obs.shape[0], -1)))
        x = self.common(x)
        return self.action(x), self.value(x)


@dataclass
class SearchResult:
    actions: list | None          # Env::solution of the best rollout, or None if none succeeded
    key: int                      # packed key of the best rollout over all ranks
    rollout_id: int               # global id of the best rollout
    success: bool
    iterations: int               # decision steps executed
    seconds: float                # wall time of the whole search incl. the reduction
    rollouts: int                 # rollouts run over all ranks


def decode_key(key: int):
    return bool((key >> KEY_SUCCESS_BIT) & 1), KEY_ID_MASK - (key & KEY_ID_MASK)


def chunk_plan(num_targets: int, targets_per_launch: int, num_rollouts: int):
    """How solve_many splits its targets: [(first target, targets in the chunk, first global rollout id)]; a chunk pads
    targets_per_launch - count slots.  Rollout ids must fit the key's 30-bit id field: num_targets * num_rollouts < 2^30."""
    if num_targets * num_rollouts >= 1 << 30:
        raise ValueError(f"{num_targets} targets x {num_rollouts} rollouts do not fit the 30-bit rollout id of the search key (< 2^30 needed)")
    return [(s, min(targets_per_launch, num_targets - s), s * num_rollouts) for s in range(0, num_targets, targets_per_launch)]


def identity_payload(env_kind: int, num_qubits: int) -> list[int]:
    """The env kind's identity as a set_state payload: a target that is solved when loaded (solve_many pads short chunks with it)."""
    n = int(num_qubits)
    if env_kind == _abi.ENV_PERMUTATION:
        return list(range(n))
    d = n if env_kind == _abi.ENV_LINEAR_FUNCTION else 2 * n
    eye = np.eye(d, dtype=np.int64).ravel().tolist()
    return [0] + eye if env_kind == _abi.ENV_PAULI_NETWORK else eye


def check_tensor_core_search(env_kind: int, num_qubits: int, num_actions: int, device=None):
    """Raises NotImplementedError where the "tensor_core" search backend cannot run: more than 127 actions (the tensor-core head), a
    Permutation wider than 64 qubits (no packed observations), a device that is not sm_100 (tcgen05)."""
    if num_actions > 127:
        raise NotImplementedError(f"the tensor-core search supports up to 127 actions (got {num_actions})")
    if env_kind == _abi.ENV_PERMUTATION and num_qubits > 64:
        raise NotImplementedError(f"the tensor-core search needs packed observations: a Permutation of {num_qubits} > 64 qubits has none")
    if not torch.cuda.is_available():
        raise RuntimeError("qiskit_gym_b200 needs a CUDA device (no CPU fallback)")
    if torch.cuda.get_device_capability(device)[0] != 10:
        raise NotImplementedError("the tensor-core search needs an sm_100 device (tcgen05)")


def check_twisted_search(env_kind: int, num_qubits: int, policy_backend: str):
    """Raises NotImplementedError where the twisted search (RolloutSearch(use_twists=True)) cannot run: the "torch" backend, PauliNetwork
    (its qubit symmetry is applied inside the env by add_perms), a Permutation wider than 64 qubits (no packed observations).  Needs no
    device."""
    if policy_backend == "torch":
        raise NotImplementedError("the twisted search runs on the packed-observation backends (persistent, fused, tensor_core), not torch")
    if env_kind == _abi.ENV_PAULI_NETWORK:
        raise NotImplementedError("PauliNetwork has no twisted search: its qubit symmetry is applied inside the env (add_perms)")
    if env_kind == _abi.ENV_PERMUTATION and num_qubits > 64:
        raise NotImplementedError(f"the twisted search needs packed observations: a Permutation of {num_qubits} > 64 qubits has none")


def twist_tables(env: BatchedEnv):
    """The env's twists (env.twists(), built with add_perms), once, on its device: uint8 [K, n] inverse qubit permutations
    (collector.qubit_twist_table) and int32 [K, A] act perms -- the tables of the twisted rollout and tree searches."""
    from .collector import qubit_twist_table
    obs_perms, act_perms = env.twists()
    qperm = torch.from_numpy(qubit_twist_table(obs_perms, int(env.cfg.num_qubits))).to(env.device)
    act = torch.from_numpy(np.asarray(act_perms, dtype=np.int32)).to(env.device)
    return qperm, act


def reduce_best(local_key: int, local_solution, group=None, device=None):
    """Cross-rank best-rollout reduction in two collectives: an all-gather of (packed key, solution length) — the owner of the winning
    rollout is the rank holding the largest key; keys are unique, they embed the global rollout id — then the owner broadcasts its action
    list.  Works with any torch.distributed backend (NCCL on GPUs, gloo in tests)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local_key, local_solution
    dev = device if device is not None else torch.device("cpu")
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sol = list(local_solution) if local_solution is not None else []
    mine = torch.tensor([local_key, len(sol)], dtype=torch.int64, device=dev)
    allk = torch.empty((world, 2), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allk, mine, group=group) if dev.type == "cuda" else dist.all_gather(list(allk.unbind(0)), mine, group=group)
    table = allk.tolist()
    best = max(k for k, _ in table)
    if best == 0:
        return 0, None
    src = next(r for r, (k, _) in enumerate(table) if k == best)       # (the lowest rank on the impossible tie)
    n = int(table[src][1])
    buf = torch.zeros(max(n, 1), dtype=torch.int64, device=dev)
    if rank == src and n:
        buf[:n] = torch.tensor(sol, dtype=torch.int64)
    dist.broadcast(buf, src=dist.get_global_rank(group, src) if group is not None else src, group=group)
    return best, [int(v) for v in buf[:n].tolist()]


def best_rollout(env: BatchedEnv):
    """(key, solution or None) of the best rollout of this rank's engine (qg_search_best)."""
    key, idx = env.search_best()
    ok, rid = decode_key(key)
    return key, (env.solution(idx) if (ok and idx >= 0) else None)


def search_result(env: BatchedEnv, key, sol, its, t0, local_rollouts, group=None, reduced=False) -> SearchResult:
    """The SearchResult of a search whose best local rollout is (key, sol): under torch.distributed, reduced over the ranks first
    (reduce_best) unless `reduced` says the key already is the global one; rollouts = local_rollouts x the world size."""
    ok, rid = decode_key(key)
    world = 1
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            world = dist.get_world_size(group)
            if not reduced:
                key, sol = reduce_best(key, sol, group=group, device=env.device if dist.get_backend(group) == "nccl" else None)
            ok, rid = decode_key(key)
    except ImportError:
        pass
    return SearchResult(actions=sol if ok else None, key=key, rollout_id=rid, success=ok, iterations=its,
                        seconds=time.perf_counter() - t0, rollouts=local_rollouts * world)


class RolloutSearch:
    """Device-resident `solve`: owns a BatchedEnv of `num_rollouts` rollouts on one GPU."""

    def __init__(self, env_kind, num_qubits, gateset, policy: torch.nn.Module, num_rollouts: int, device=None,
                 max_depth: int = 128, use_cuda_graph: bool = True, policy_backend: str = "persistent", targets_per_launch: int = 1,
                 use_twists: bool = False, **env_kwargs):
        """policy_backend: "persistent" = the whole search in ONE kernel launch (qg_search_run: every CTA loops policy -> sample ->
        step for its 8 rollouts); "fused" = two launches per decision (policy.FusedPolicy + qg_search_step_bits) in a CUDA graph;
        "torch" = dense f32 observations + the PyTorch module (cuBLAS GEMMs, softmax).  "persistent" and "fused" take identical
        decisions (same kernels' device code, same bits).
        "tensor_core" = the "fused" decision with the policy on tcgen05 tensor cores (policy.TensorCorePolicy with max_batch = the
        engine's rollouts, no value head): observe bits -> qg_policy_tc_forward_bits -> qg_search_step_bits, in a CUDA graph.  It is
        built for large batches (solve_many at tens of thousands of rollouts per launch) and is opt-in: its f16 hi+lo split arithmetic
        rounds differently from the f32 backends, so its decisions are not theirs (the probabilities are within TensorCorePolicy's error
        bound of the float64 module).  Each row's probabilities are bit-identical whatever the batch size and the other rows, so the
        solve_many contract below holds among "tensor_core" searches.  NotImplementedError where it cannot run: more than 127 actions,
        a Permutation wider than 64 qubits (no packed observations), a device that is not sm_100.
        Every search starts by refreshing the policy handle from `self.policy` (policy.FusedPolicy / TensorCorePolicy.refresh): a weight
        update (optimizer step, load_state_dict) or another module assigned to `policy` is what the next search runs.  "tensor_core" copies
        a weight update into the handle in place (captured graphs stay valid).
        targets_per_launch: solve_many searches that many targets together, each with its own `num_rollouts` rollouts (the engine
        holds targets_per_launch * num_rollouts); solve() needs targets_per_launch == 1.
        use_twists: the twisted search (include/qg_engine.h qg_search_run_twisted): every rollout runs the policy, at every decision, in a
        symmetry frame of the env (its twists() with add_perms, as the collector trains it) drawn from the seed, the rollout's global id
        and the decision index; the env's actions are weighed through the frame's act perm.  Backends "persistent", "fused" and
        "tensor_core"; Permutation (<= 64 qubits), LinearFunction and Clifford.  NotImplementedError, before anything is allocated, for
        "torch", PauliNetwork (its symmetry is applied inside the env) and a Permutation wider than 64 qubits."""
        if targets_per_launch < 1:
            raise ValueError("targets_per_launch must be >= 1")
        assert policy_backend in ("persistent", "fused", "torch", "tensor_core")
        if use_twists:
            check_twisted_search(env_kind, num_qubits, policy_backend)
            if env_kwargs.get("add_perms") is False:
                raise ValueError("use_twists needs the env's twists: add_perms=False contradicts it")
            env_kwargs["add_perms"] = True
        env_kwargs.setdefault("add_perms", False)
        self.env_kind, self.num_qubits = env_kind, num_qubits
        self.R, self.targets_per_launch = num_rollouts, targets_per_launch
        self.env = BatchedEnv(env_kind, num_qubits, gateset, targets_per_launch * num_rollouts, device=device, max_depth=max_depth, **env_kwargs)
        self.policy = policy.to(self.env.device).eval()
        self.backend = policy_backend
        self.max_depth = max_depth
        self.B = targets_per_launch * num_rollouts
        dev = self.env.device
        self.handle = None          # the policy's C handle (policy.FusedPolicy / TensorCorePolicy); None for "torch"
        if policy_backend in ("fused", "persistent"):
            from .policy import FusedPolicy
            self.handle = FusedPolicy(self.policy, device=dev)
        if policy_backend == "tensor_core":
            from .policy import TensorCorePolicy
            check_tensor_core_search(env_kind, num_qubits, self.env.num_actions(), dev)
            self.handle = TensorCorePolicy(self.policy, max_batch=self.B, device=dev, with_value=False)
        if policy_backend != "torch":
            self.obs_bits = self.env.new_obs_bits()
        self.probs = torch.zeros((self.B, self.env.num_actions()), dtype=torch.float32, device=dev)
        self.num_active = torch.zeros(1, dtype=torch.int32, device=dev)
        self.use_twists = bool(use_twists)
        self.qperm_table = self.act_table = self.twist = None
        if self.use_twists:
            self.qperm_table, self.act_table = twist_tables(self.env)
            self.twist = torch.zeros(self.B, dtype=torch.int32, device=dev)
        self.num_twists = 0 if self.qperm_table is None else int(self.qperm_table.shape[0])
        self.use_graph = use_cuda_graph
        self.hook = None            # tests: hook(probs, obs_bits) sees every decision's policy output before the step reads it (no graph);
                                    # twisted searches call hook(probs, obs_bits, twist) with the decision's frames
        self._graphs = {}
        self._stream = torch.cuda.Stream(device=dev)
        self._decisions = torch.zeros((self.B + 7) // 8, dtype=torch.int32, device=dev)

    # the handle under the names it had per backend before `handle` (read by existing callers): None for the other backends
    fused = property(lambda self: self.handle if self.backend in ("fused", "persistent") else None)
    tcp = property(lambda self: self.handle if self.backend == "tensor_core" else None)

    def check_supported(self):
        """Raises NotImplementedError (QG_ERR_UNSUPPORTED) now rather than in the first solve() when the one-launch search cannot run
        this env / policy pair: a zero-decision qg_search_run goes through all of its checks without launching anything."""
        if self.backend == "persistent":
            self._run(0, True)

    def _run(self, max_decisions, deterministic):
        if self.use_twists:
            self.env.search_run_twisted(self.handle, self.obs_bits, self.probs, max_decisions, self.qperm_table, self.act_table, self.twist,
                                        deterministic=deterministic, decisions=self._decisions)
        else:
            self.env.search_run(self.handle, self.obs_bits, self.probs, max_decisions, deterministic=deterministic, decisions=self._decisions)

    def _iteration(self, deterministic):
        if self.backend in ("fused", "tensor_core"):
            self.handle.forward_bits(self.obs_bits, probs=self.probs)
            if self.use_twists:
                if self.hook is not None:
                    self.hook(self.probs, self.obs_bits, self.twist)
                self.env.search_step_twisted(self.probs, self.obs_bits, self.qperm_table, self.act_table, self.twist, deterministic=deterministic,
                                             num_active=self.num_active)
                return
            if self.hook is not None:
                self.hook(self.probs, self.obs_bits)
            self.env.search_step_bits(self.probs, self.obs_bits, deterministic=deterministic, num_active=self.num_active)
            return
        with torch.no_grad():
            logits, _ = self.policy(self.env.obs)
            torch.softmax(logits.float(), dim=-1, out=self.probs)
        self.env.search_step(self.probs, deterministic=deterministic, obs=True, num_active=self.num_active)

    def _observe(self):
        if self.use_twists:
            self.env.search_observe_twisted(self.obs_bits, self.qperm_table, self.twist)
        elif self.backend != "torch":
            self.env.observe_bits(self.obs_bits)
        else:
            self.env.observe()

    def _refresh_weights(self, caller):
        """Brings the handle up to self.policy; runs on self._stream, whose refresh work waits for the caller's stream.  A recreated
        handle drops the graphs captured with the old one."""
        if self.handle is not None and self.handle.refresh(self.policy, after=caller):
            self._graphs = {}

    def _graph(self, deterministic, params):
        """The CUDA graph of one iteration.  Its launches carry the engine's seed and first rollout id as they were at capture (the
        step kernel takes them by value), so a graph serves only searches with the same (seed, first rollout id): `params`."""
        g, captured = self._graphs.get(deterministic, (None, None))
        if g is None or captured != params:
            # warm-up outside capture (cuBLAS workspaces, lazy module init), on a scratch copy of the state
            self.env.snapshot()
            for _ in range(2):
                self._iteration(deterministic)
            self.env.restore()
            torch.cuda.current_stream(self.env.device).synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self._stream):
                self._iteration(deterministic)
            self.env.restore()
            self._graphs[deterministic] = (g, params)
        return g

    def _search(self, load, deterministic, seed, first_rollout_id, check_every):
        """One search on self._stream (the caller enters it): load() puts the targets into the rollouts, then the decisions run.
        Returns the number of decision steps, or None for the one-launch search (its CTAs' counts are in self._decisions)."""
        env = self.env
        if self.backend == "persistent":
            load()
            env.search_begin(seed, first_rollout_id)
            self._observe()
            self._run(self.max_depth, deterministic)
            return None
        load()
        use_graph = self.use_graph and self.hook is None
        if use_graph:
            env.search_begin(seed, first_rollout_id)        # (what the captured launches see)
            g = self._graph(deterministic, (seed, first_rollout_id))
            load()
        env.search_begin(seed, first_rollout_id)
        self._observe()
        its = 0
        while its < self.max_depth:
            if use_graph:
                g.replay()
            else:
                self._iteration(deterministic)
            its += 1
            if its % check_every == 0 and int(self.num_active.item()) == 0:
                break
        return its

    def solve(self, state, deterministic: bool = False, seed: int = 0, first_rollout_id: int = 0, check_every: int = 8,
              group=None, comm=None) -> SearchResult:
        """group: torch.distributed group for the Python-side cross-rank reduction (reduce_best); comm: an ncclComm_t handle for the
        C-side one (qg_search_finish); with neither, and torch.distributed initialised, the default group is used."""
        if self.targets_per_launch != 1:
            raise ValueError("solve() searches one target: use solve_many() on a search built with targets_per_launch > 1")
        env = self.env
        t0 = time.perf_counter()
        caller = torch.cuda.current_stream(env.device)
        with torch.cuda.stream(self._stream):
            self._refresh_weights(caller)
            # broadcast: every rollout starts from the target
            its = self._search(lambda: env.set_state(state), deterministic, seed, first_rollout_id, check_every)
            if comm is not None:        # qg_search_finish reduces over ALL ranks itself (one all-gather + on-GPU pick), no torch collective
                key, ok, rid, owner, sol = env.search_finish(comm)
            else:
                key, sol = best_rollout(env)
            if its is None:
                its = int(self._decisions.max().item())
        return search_result(env, key, sol, its, t0, self.B, group, reduced=comm is not None)

    def solve_many(self, states, deterministic: bool = False, seed: int = 0, check_every: int = 8) -> list[SearchResult]:
        """solve() for many targets, targets_per_launch of them per search.  Target t gets global rollout ids t*R .. t*R + R - 1
        (R = num_rollouts), so its result equals solve(states[t], deterministic, seed, first_rollout_id=t*R) of a single-target search
        with the same policy and backend, whatever targets_per_launch is.  A short last chunk fills its free slots with the env kind's
        identity, which is final when loaded.  Each chunk: grouped load, the search, the per-target winner reduction on the device and
        one device-to-host copy.  SearchResult.seconds is the chunk's wall time, .rollouts = R."""
        states = list(states)
        T, R = self.targets_per_launch, self.R
        plan = chunk_plan(len(states), T, R)
        env = self.env
        cap = max(int(env.cfg.solution_capacity) or (self.max_depth + 16), 1)
        words = T * (3 + cap) + 1                           # keys (2 words each), lengths, action rows, decision count
        if getattr(self, "_win", None) is None or self._win.numel() != words:
            self._win = torch.zeros(words, dtype=torch.int32, device=env.device)
            self._win_host = torch.zeros(words, dtype=torch.int32, pin_memory=True)
        pad = identity_payload(self.env_kind, self.num_qubits)
        caller = torch.cuda.current_stream(env.device)
        with torch.cuda.stream(self._stream):
            self._refresh_weights(caller)
        out = []
        for start, count, first_id in plan:
            t0 = time.perf_counter()
            chunk = states[start: start + count] + [pad] * (T - count)
            with torch.cuda.stream(self._stream):
                its = self._search(lambda: env.set_state_grouped(chunk, R), deterministic, seed, first_id, check_every)
                env.search_best_grouped(R, T, cap, out=self._win[: words - 1])
                if its is None:
                    torch.amax(self._decisions, dim=0, keepdim=True, out=self._win[words - 1:])
                self._win_host.copy_(self._win, non_blocking=True)
                self._stream.synchronize()
            h = self._win_host.numpy()
            keys, lens, rows = h[: 2 * T].view(np.int64), h[2 * T: 3 * T], h[3 * T: words - 1].view(np.uint32).reshape(T, cap)
            if its is None:
                its = int(h[words - 1])
            dt = time.perf_counter() - t0
            for j in range(count):
                key = int(keys[j])
                ok, rid = decode_key(key)
                if ok and lens[j] < 0:
                    raise ValueError(f"a solution is longer than cap={cap}")
                out.append(SearchResult(actions=rows[j, : lens[j]].astype(np.int64).tolist() if ok else None, key=key, rollout_id=rid,
                                        success=ok, iterations=its, seconds=dt, rollouts=R))
        return out
