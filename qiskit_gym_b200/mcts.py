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
from .search import SearchResult, best_rollout, search_result


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


class MCTSSearch:
    """`solve` with a tree search per decision.  Owns the rollout engine (R envs, solutions tracked) and a slot-pool engine of
    R * node_cap records for the tree nodes (node_cap = num_mcts_searches + 1, or 2 * num_mcts_searches + 1 with reuse_tree)."""

    def __init__(self, env_kind, num_qubits, gateset, policy: torch.nn.Module, num_rollouts: int, num_mcts_searches: int, C: float = 2 ** 0.5,
                 device=None, max_depth: int = 128, use_cuda_graph: bool = True, policy_backend: str = "auto", reuse_tree: bool = False,
                 **env_kwargs):
        """use_cuda_graph: a decision's launches (root evaluation, then per simulation PUCT descent -> clone + step -> policy -> back-up)
        are captured once and replayed: the whole decision as one graph up to 128 simulations, one graph per simulation beyond.
        policy_backend: "fused" = priors and values of the root / the leaves from packed observations in one kernel (policy.FusedPolicy
        with the value head, refreshed from `policy` before every decision), "torch" = the PyTorch module on dense observations, "auto" =
        fused when the policy has the simple head layout and the env can pack its observations.
        reuse_tree: each decision after the first of a `solve` keeps up to num_mcts_searches + 1 nodes of the subtree below the action
        the rollout played, with their statistics, and adds num_mcts_searches simulations to them (qg_mcts_reroot).  The rollout's
        action must then reach `decide` through `chosen` (solve does it; a caller driving decide itself passes chosen=self.chosen
        to search_step).  `reused[i]` tells whether tree i was kept at the last decision."""
        assert num_mcts_searches >= 1 and policy_backend in ("auto", "fused", "torch")
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
        self.hook = None            # tests: hook(kind, decision, simulation, tensors...) sees the policy outputs the trees consumed
        from .policy import FusedPolicy, simple_value_head
        can_fuse = simple_value_head(self.policy) is not None and not (env_kind == 0 and num_qubits > 64)      # (no packed observations for n > 64 permutations)
        if policy_backend == "fused" and not can_fuse:
            raise NotImplementedError("policy_backend='fused' needs single-Linear action / value heads")
        self.backend = "fused" if (policy_backend != "torch" and can_fuse) else "torch"
        self.fused = None
        if self.backend == "fused":
            self.root_bits = self.env.new_obs_bits()
            self.leaf_bits = torch.zeros((self.R, self.env.obs_words()), dtype=torch.int32, device=dev)
            self.pri = torch.zeros((self.R, A), dtype=torch.float32, device=dev)
            self.val = torch.zeros(self.R, dtype=torch.float32, device=dev)
            self.fused = FusedPolicy(self.policy, device=dev, with_value=True)
        self.use_graph = bool(use_cuda_graph)
        self._graphs = None         # (module captured, root graph or None, simulation graph or None, whole-decision graph or None)
        self._stream = torch.cuda.Stream(device=dev)

    def _policy(self, obs):
        with torch.no_grad():
            logits, value = self.policy(obs)
            return torch.softmax(logits.float(), dim=-1).contiguous(), value.float().reshape(-1).contiguous()

    def _root(self, decision: int = 0):
        env, pool, tree = self.env, self.pool, self.tree
        if self.reuse:
            tree.reroot(pool, env, self.chosen, self.NC - self.S, self.reused)
        _, done, _, _ = env.status()
        if self.backend == "fused":
            env.observe_bits(self.root_bits)
            self.fused.forward_bits(self.root_bits, probs=self.pri, values=self.val)
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
        if self.backend == "fused":
            pool.step_slots(self.src, self.dst, self.act, obs_bits=self.leaf_bits, reward=self.leaf_reward, done=self.leaf_done)
            self.fused.forward_bits(self.leaf_bits, probs=self.pri, values=self.val)
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
        if (self.fused is not None and self.fused.refresh(self.policy)) or (self._graphs is not None and self._graphs[0] is not self.policy):
            self._graphs = None
        fresh, self._fresh = self._fresh, False
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
