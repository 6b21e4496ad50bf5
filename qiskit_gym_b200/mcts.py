"""Batched PUCT tree search on the device (SURVEY.md §8f row 4): the `num_mcts_searches > 0` branch of the reference's
`algorithm.solve(state, deterministic, num_searches, num_mcts_searches, C, max_expand_depth)` (rl/synthesis.py:122-124;
rl/configs.py:30-42 documents the knobs).

`num_searches` rollouts run side by side as in search.RolloutSearch; before each decision every rollout grows its own tree
of `num_mcts_searches` simulations from its current env state, and the decision is drawn from the root's visit counts
instead of the raw policy output.  The tree bookkeeping (PUCT descent, node creation, return back-up) is csrc/qg_mcts.cu;
a child node's env is the parent's record cloned and stepped in one pass through a pool of record slots
(`qg_step_slots`); the policy evaluates all new leaves of a simulation round in one batch.

With `reuse_tree=True` a decision starts from the subtree below the action the rollout played (AlphaGo Zero's tree reuse), kept
when the tree's node for it holds the env the rollout reached (csrc/qg_mcts.cu states the rule).

With `policy_backend="tensor_core"` the roots and leaves are evaluated by the tcgen05 tensor-core policy (policy.TensorCorePolicy) instead of
the f32 FFMA kernel: opt-in, for searches over thousands of trees, where the FFMA policy is what a simulation waits for.

With `use_twists=True` every policy evaluation of a tree (its root, each new leaf) runs in a symmetry frame of the env drawn per
rollout, decision and evaluation, the way the collector trains the policy; the trees keep their priors in env action order
(csrc/qg_mcts.cu states the protocol).

twisterl's own tree search is not in the reference tree: the protocol (stated in csrc/qg_mcts.cu) is this engine's, and
`max_expand_depth` — whose exact meaning cannot be recovered from the reference — is accepted and must be 1.
"""
from __future__ import annotations

import ctypes as C
import time

import torch

from . import _abi
from ._lib import check, lib
from .engine import BatchedEnv, _dptr
from .search import SearchResult, best_rollout, check_tensor_core_search, check_twisted_search, search_result, twist_tables


class TreeArrays:
    """Device arrays of `num_trees` trees with `node_cap` nodes (qg_mcts_tree)."""

    def __init__(self, num_trees: int, node_cap: int, num_actions: int, device):
        R, NC, A = num_trees, node_cap, num_actions
        f32, i32 = torch.float32, torch.int32
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=device)
        self.prior, self.visits, self.value_sum, self.child = z((R, NC, A), f32), z((R, NC, A), i32), z((R, NC, A), f32), z((R, NC, A), i32)
        self.node_reward, self.node_final, self.node_count = z((R, NC), f32), z((R, NC), torch.uint8), z((R,), i32)
        self.path_node, self.path_action, self.path_len, self.new_node = z((R, NC), i32), z((R, NC), i32), z((R,), i32), z((R,), i32)
        self.c = _abi.QgMctsTree(R, NC, A, *[t.data_ptr() for t in (self.prior, self.visits, self.value_sum, self.child, self.node_reward, self.node_final,
                                                                     self.node_count, self.path_node, self.path_action, self.path_len, self.new_node)])
        self.device = device

    def _st(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def begin(self, root_prior, root_final):
        check(lib().qg_mcts_begin(C.byref(self.c), _dptr(root_prior), _dptr(root_final), self._st()))

    def select(self, c_puct, src_slot, dst_slot, action):
        check(lib().qg_mcts_select(C.byref(self.c), C.c_float(c_puct), _dptr(src_slot), _dptr(dst_slot), _dptr(action), self._st()))

    def backup(self, prior, value, reward, done):
        check(lib().qg_mcts_backup(C.byref(self.c), _dptr(prior), _dptr(value), _dptr(reward), _dptr(done), self._st()))

    def root_weights(self, out):
        check(lib().qg_mcts_root_weights(C.byref(self.c), _dptr(out), self._st()))
        return out

    def reroot(self, pool, rollouts, chosen, keep_nodes, reused):
        check(lib().qg_mcts_reroot(C.byref(self.c), pool._h, rollouts._h, _dptr(chosen), int(keep_nodes), _dptr(reused), self._st()))

    def begin_keep(self, root_prior, root_final, reused):
        check(lib().qg_mcts_begin_keep(C.byref(self.c), _dptr(root_prior), _dptr(root_final), _dptr(reused), self._st()))

    # the twisted forms: priors in the policy's frame twist[i] (act_table int32 [K, A]), stored in env action order
    def begin_twisted(self, root_prior, root_final, act_table, twist, reused=None):
        K = int(act_table.shape[0])
        if reused is None:
            check(lib().qg_mcts_begin_twisted(C.byref(self.c), _dptr(root_prior), _dptr(root_final), _dptr(act_table), K, _dptr(twist), self._st()))
        else:
            check(lib().qg_mcts_begin_keep_twisted(C.byref(self.c), _dptr(root_prior), _dptr(root_final), _dptr(reused), _dptr(act_table), K,
                                                   _dptr(twist), self._st()))

    def backup_twisted(self, prior, value, reward, done, act_table, twist, eval_index):
        check(lib().qg_mcts_backup_twisted(C.byref(self.c), _dptr(prior), _dptr(value), _dptr(reward), _dptr(done), _dptr(act_table),
                                           int(act_table.shape[0]), _dptr(twist), _dptr(eval_index), self._st()))


def observe_twisted(rollouts: BatchedEnv, pool: BatchedEnv | None, dst_slot, action, search_key, eval_index, qperm_table, obs_bits, twist):
    """qg_mcts_observe_twisted: the root pass (pool None) or the leaf pass of the twisted tree search -> packed bits obs_bits int32
    [R, obs_words] and frames twist int32 [R].  search_key int64 [2] = (seed, first rollout id), eval_index int32 [1]: device memory."""
    check(lib().qg_mcts_observe_twisted(rollouts._h, None if pool is None else pool._h, _dptr(dst_slot), _dptr(action), _dptr(search_key),
                                        _dptr(eval_index), _dptr(qperm_table), int(qperm_table.shape[0]), _dptr(obs_bits), _dptr(twist),
                                        rollouts._stream()))


def check_twisted_tree_search(env_kind: int, num_qubits: int, policy: torch.nn.Module, policy_backend: str, env_kwargs: dict):
    """Raises, before anything is allocated, where the twisted tree search cannot run: NotImplementedError for the "torch" backend, a
    policy without single-Linear action / value heads (nothing fused to run), PauliNetwork and a Permutation wider than 64 qubits;
    ValueError for an explicit add_perms=False."""
    from .policy import simple_value_head
    if policy_backend == "torch":
        raise NotImplementedError("the twisted tree search evaluates packed observations on the fused policy, not the torch backend")
    check_twisted_search(env_kind, num_qubits, "fused")
    if simple_value_head(policy) is None:
        raise NotImplementedError("the twisted tree search runs the fused policy: it needs single-Linear action / value heads")
    if env_kwargs.get("add_perms") is False:
        raise ValueError("use_twists needs the env's twists: add_perms=False contradicts it")


def check_tensor_core_tree_search(env_kind: int, num_qubits: int, num_actions: int, policy: torch.nn.Module, device=None):
    """Raises NotImplementedError, before anything is allocated, where the "tensor_core" tree search cannot run: the tensor-core search's
    limits (search.check_tensor_core_search) and a policy without single-Linear action / value heads (the trees need the value head)."""
    from .policy import simple_value_head
    if simple_value_head(policy) is None:
        raise NotImplementedError("the tensor-core tree search evaluates the value head with the policy: it needs single-Linear action / value heads")
    check_tensor_core_search(env_kind, num_qubits, num_actions, device)


class MCTSSearch:
    """`solve` with a tree search per decision.  Owns the rollout engine (R envs, solutions tracked) and a slot-pool engine of
    R * node_cap records for the tree nodes (node_cap = num_mcts_searches + 1, or 2 * num_mcts_searches + 1 with reuse_tree)."""

    def __init__(self, env_kind, num_qubits, gateset, policy: torch.nn.Module, num_rollouts: int, num_mcts_searches: int, C: float = 2 ** 0.5,
                 device=None, max_depth: int = 128, use_cuda_graph: bool = True, policy_backend: str = "auto", reuse_tree: bool = False,
                 use_twists: bool = False, **env_kwargs):
        """use_cuda_graph: a decision's launches (root evaluation, then per simulation PUCT descent -> clone + step -> policy -> back-up)
        are captured once and replayed: the whole decision as one graph up to 128 simulations, one graph per simulation beyond.
        policy_backend: "fused" = priors and values of the root / the leaves from packed observations in one kernel (policy.FusedPolicy
        with the value head, refreshed from `policy` before every decision), "torch" = the PyTorch module on dense observations, "auto" =
        fused when the policy has the simple head layout and the env can pack its observations.  "tensor_core" = the "fused" decision with
        the priors and values from the tcgen05 tensor-core policy (policy.TensorCorePolicy with max_batch = num_rollouts and the value
        head) on the same packed observations; built for searches over thousands of trees.  It is opt-in and never chosen by "auto": its
        f16 hi+lo split arithmetic rounds differently from the f32 backends, so its trees are not theirs (priors and values within
        TensorCorePolicy's error bound of the float64 module).  Each row's outputs are bit-identical whatever the batch, so a tree's
        search does not depend on how many trees share the launch.  NotImplementedError, before anything is allocated, where it cannot
        run: more than 127 actions, a Permutation wider than 64 qubits, a device that is not sm_100 (search.check_tensor_core_search),
        a policy without single-Linear action / value heads.
        Every decision starts by refreshing the policy handle from `self.policy`: "fused" recreates it on a weight change (the decision
        graphs are captured again), "tensor_core" loads a weight update (optimizer step, load_state_dict) in place, so the captured
        graphs stay valid and replay the new weights.
        reuse_tree: each decision after the first of a `solve` keeps up to num_mcts_searches + 1 nodes of the subtree below the action
        the rollout played, with their statistics, and adds num_mcts_searches simulations to them (qg_mcts_reroot).  The rollout's
        action must then reach `decide` through `chosen` (solve does it; a caller driving decide itself passes chosen=self.chosen
        to search_step).  `reused[i]` tells whether tree i was kept at the last decision.
        use_twists: the twisted tree search (include/qg_engine.h qg_mcts_observe_twisted): the root and every new leaf are evaluated in
        a symmetry frame of the env (its twists() with add_perms) drawn from the seed and first rollout id of env.search_begin, the
        rollout's global id, its step counter and the evaluation index; the node stores P(a) = probs[act_perm[k][a]].  Runs on the fused
        and "tensor_core" backends; `root_twist` holds the root frames of the last decision and `root_bits` the twisted root
        observations.  Raises before anything is allocated where it cannot run (check_twisted_tree_search)."""
        assert num_mcts_searches >= 1 and policy_backend in ("auto", "fused", "torch", "tensor_core")
        if use_twists:
            check_twisted_tree_search(env_kind, num_qubits, policy, policy_backend, env_kwargs)
            env_kwargs["add_perms"] = True
        if policy_backend == "tensor_core":
            check_tensor_core_tree_search(env_kind, num_qubits, len(gateset), policy, device)
        env_kwargs.setdefault("add_perms", False)
        self.env = BatchedEnv(env_kind, num_qubits, gateset, num_rollouts, device=device, max_depth=max_depth, **env_kwargs)
        pool_kwargs = dict(env_kwargs, track_solution=False)
        self.reuse = bool(reuse_tree)
        self.S, self.R = int(num_mcts_searches), int(num_rollouts)
        self.NC = (2 * self.S + 1) if self.reuse else (self.S + 1)
        self.pool = BatchedEnv(env_kind, num_qubits, gateset, self.R * self.NC, device=self.env.device_index, max_depth=max_depth, **pool_kwargs)
        self.policy = policy.to(self.env.device).eval()
        self.c_puct, self.max_depth = float(C), int(max_depth)
        dev = self.env.device
        A = self.env.num_actions()
        self.tree = TreeArrays(self.R, self.NC, A, dev)
        i32 = torch.int32
        self.root_slots = (torch.arange(self.R, device=dev, dtype=torch.int64) * self.NC).to(i32)
        self.src, self.dst, self.act = (torch.zeros(self.R, dtype=i32, device=dev) for _ in range(3))
        self.leaf_obs = torch.zeros((self.R,) + tuple(self.env.obs_shape()), dtype=torch.float32, device=dev)
        self.leaf_reward = torch.zeros(self.R, dtype=torch.float32, device=dev)
        self.leaf_done = torch.zeros(self.R, dtype=torch.bool, device=dev)
        self.weights = torch.zeros((self.R, A), dtype=torch.float32, device=dev)
        self.chosen = torch.full((self.R,), -1, dtype=i32, device=dev)        # the rollouts' last actions (-1: none, fresh trees)
        self.reused = torch.zeros(self.R, dtype=torch.uint8, device=dev)       # 1: tree i was re-rooted at the last decision
        self._fresh = True          # chosen is all -1: the next decision starts every tree afresh
        self.num_active = torch.zeros(1, dtype=torch.int32, device=dev)
        self.hook = None            # tests: hook(kind, decision, simulation, prior, value) sees the policy outputs the trees consumed;
                                    # twisted searches call hook(kind, decision, simulation, prior, value, frames, obs_bits)
        from .policy import FusedPolicy, TensorCorePolicy, simple_value_head
        can_fuse = simple_value_head(self.policy) is not None and not (env_kind == 0 and num_qubits > 64)      # (no packed observations for n > 64 permutations)
        if policy_backend == "fused" and not can_fuse:
            raise NotImplementedError("policy_backend='fused' needs single-Linear action / value heads")
        if policy_backend == "tensor_core":
            self.backend = "tensor_core"
        else:
            self.backend = "fused" if (policy_backend != "torch" and can_fuse) else "torch"
        self.handle = None          # the policy's C handle (policy.FusedPolicy / TensorCorePolicy); None for "torch"
        if self.backend != "torch":
            self.root_bits = self.env.new_obs_bits()
            self.leaf_bits = torch.zeros((self.R, self.env.obs_words()), dtype=torch.int32, device=dev)
            self.pri = torch.zeros((self.R, A), dtype=torch.float32, device=dev)
            self.val = torch.zeros(self.R, dtype=torch.float32, device=dev)
            if self.backend == "fused":
                self.handle = FusedPolicy(self.policy, device=dev, with_value=True)
            else:
                self.handle = TensorCorePolicy(self.policy, max_batch=self.R, device=dev, with_value=True)
        self.use_twists = bool(use_twists)
        self.num_twists = 0
        if self.use_twists:
            self.qperm_table, self.act_table = twist_tables(self.env)
            self.num_twists = int(self.act_table.shape[0])
            self.root_twist = torch.zeros(self.R, dtype=i32, device=dev)      # frames of the root evaluations of the last decision
            self.leaf_twist = torch.zeros(self.R, dtype=i32, device=dev)      # frames of the last simulation's leaf evaluations
            self.search_key = torch.zeros(2, dtype=torch.int64, device=dev)   # (seed, first rollout id) of env.search_begin, read by the kernels
            self.eval_index = torch.zeros(1, dtype=i32, device=dev)           # evaluation index - 1 (reset by the root pass, advanced by back-up)
            self._key = None
        self.use_graph = bool(use_cuda_graph)
        self._graphs = None         # (module captured, root graph or None, simulation graph or None, whole-decision graph or None)
        self._stream = torch.cuda.Stream(device=dev)

    # the handle under the name it had before `handle` (read by existing callers): None for the other backends
    fused = property(lambda self: self.handle if self.backend == "fused" else None)

    def _policy(self, obs):
        with torch.no_grad():
            logits, value = self.policy(obs)
            return torch.softmax(logits.float(), dim=-1).contiguous(), value.float().reshape(-1).contiguous()

    def _root(self, decision: int = 0):
        env, pool, tree = self.env, self.pool, self.tree
        if self.reuse:
            tree.reroot(pool, env, self.chosen, self.NC - self.S, self.reused)
        _, done, _, _ = env.status()
        if self.use_twists:
            observe_twisted(env, None, None, None, self.search_key, self.eval_index, self.qperm_table, self.root_bits, self.root_twist)
            self.handle.forward_bits(self.root_bits, probs=self.pri, values=self.val)
            if self.hook:
                self.hook("root", decision, -1, self.pri, None, self.root_twist, self.root_bits)
            pool.copy_records_from(env, self.root_slots)
            tree.begin_twisted(self.pri, done, self.act_table, self.root_twist, self.reused if self.reuse else None)
            return
        if self.backend != "torch":
            env.observe_bits(self.root_bits)
            self.handle.forward_bits(self.root_bits, probs=self.pri, values=self.val)
            prior = self.pri
        else:
            env.observe()
            prior, _ = self._policy(env.obs)
        if self.hook:
            self.hook("root", decision, -1, prior, None)
        pool.copy_records_from(env, self.root_slots)          # (a re-rooted tree's root record already equals it)
        if self.reuse:
            tree.begin_keep(prior, done, self.reused)
        else:
            tree.begin(prior, done)

    def _simulation(self, decision: int = 0, s: int = 0):
        pool, tree = self.pool, self.tree
        tree.select(self.c_puct, self.src, self.dst, self.act)
        if self.use_twists:
            pool.step_slots(self.src, self.dst, self.act, reward=self.leaf_reward, done=self.leaf_done)
            observe_twisted(self.env, pool, self.dst, self.act, self.search_key, self.eval_index, self.qperm_table, self.leaf_bits, self.leaf_twist)
            self.handle.forward_bits(self.leaf_bits, probs=self.pri, values=self.val)
            if self.hook:
                self.hook("leaf", decision, s, self.pri, self.val, self.leaf_twist, self.leaf_bits)
            tree.backup_twisted(self.pri, self.val, self.leaf_reward, self.leaf_done, self.act_table, self.leaf_twist, self.eval_index)
            return
        if self.backend != "torch":
            pool.step_slots(self.src, self.dst, self.act, obs_bits=self.leaf_bits, reward=self.leaf_reward, done=self.leaf_done)
            self.handle.forward_bits(self.leaf_bits, probs=self.pri, values=self.val)
            p, v = self.pri, self.val
        else:
            pool.step_slots(self.src, self.dst, self.act, obs=self.leaf_obs, reward=self.leaf_reward, done=self.leaf_done)
            p, v = self._policy(self.leaf_obs)
        if self.hook:
            self.hook("leaf", decision, s, p, v)
        tree.backup(p, v, self.leaf_reward, self.leaf_done)

    def _decide_eager(self, decision: int = 0):
        self._root(decision)
        for s in range(self.S):
            self._simulation(decision, s)
        return self.tree.root_weights(self.weights)

    def _capture(self):
        """Graphs of one decision.  The search reads the rollout engine and writes only the slot pool, the trees and self.weights, so
        the warm-up runs (cuBLAS workspaces, lazy initialisation) leave the rollouts untouched.  With reuse_tree they would overwrite
        trees that the next decision keeps: decide() captures only while every tree starts afresh (chosen all -1)."""
        dev = self.env.device
        for _ in range(2):
            self._root()
            self._simulation()
        self.tree.root_weights(self.weights)
        torch.cuda.current_stream(dev).synchronize()
        if self.S <= 128:
            whole = torch.cuda.CUDAGraph()
            with torch.cuda.graph(whole, stream=self._stream):
                self._decide_eager()
            self._graphs = (self.policy, None, None, whole)
        else:
            root, sim = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(root, stream=self._stream):
                self._root()
            with torch.cuda.graph(sim, stream=self._stream):
                self._simulation()
            self._graphs = (self.policy, root, sim, None)

    def decide(self, decision: int = 0):
        """One decision's tree search for every rollout; leaves the root visit weights in self.weights."""
        # a graph holds the policy handle and the module's parameter tensors
        if (self.handle is not None and self.handle.refresh(self.policy)) or (self._graphs is not None and self._graphs[0] is not self.policy):
            self._graphs = None
        fresh, self._fresh = self._fresh, False
        if self.use_twists and self._key != self.env.search_key:
            # read by the kernels at run time, so the captured graphs serve every seed; written outside them, on the caller's stream
            # (fills carry the values as kernel arguments: no host synchronisation)
            seed, first = self.env.search_key
            self.search_key[0].fill_(seed - (1 << 64) if seed >= (1 << 63) else seed)
            self.search_key[1].fill_(first)
            self._key = self.env.search_key
        if not self.use_graph or self.hook is not None:
            return self._decide_eager(decision)
        if self._graphs is None:
            if self.reuse and not fresh:
                return self._decide_eager(decision)
            self._capture()
        _, root, sim, whole = self._graphs
        if whole is not None:
            whole.replay()
            return self.weights
        root.replay()
        for _ in range(self.S):
            sim.replay()
        return self.tree.root_weights(self.weights)

    def solve(self, state, deterministic: bool = False, seed: int = 0, first_rollout_id: int = 0, check_every: int = 4, group=None) -> SearchResult:
        env = self.env
        t0 = time.perf_counter()
        env.set_state(state)
        env.search_begin(seed, first_rollout_id)
        self.chosen.fill_(-1)
        self._fresh = True
        its = 0
        while its < self.max_depth:
            self.decide(its)
            env.search_step(self.weights, deterministic=deterministic, obs=False, chosen=self.chosen, num_active=self.num_active)
            its += 1
            if its % check_every == 0 and int(self.num_active.item()) == 0:
                break
        key, sol = best_rollout(env)
        return search_result(env, key, sol, its, t0, self.R, group)
