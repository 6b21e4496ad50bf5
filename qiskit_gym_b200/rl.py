"""`RLSynthesis` over the device-resident search (reference src/qiskit_gym/rl/synthesis.py:32-147).

The reference builds a twisterl algorithm object around the raw env and calls `algorithm.solve(state,
deterministic, num_searches, num_mcts_searches, C, max_expand_depth)` (112-126).  Here `solve` is
`search.RolloutSearch`: `num_searches` policy-guided rollouts stepped together on the GPU, the best one reduced on
the device (and across ranks).  Config files and checkpoints are the reference's own formats: the `.json` written by
`RLSynthesis.save` (79-93) and the policy `state_dict` `.pt` (examples/models/*), so models trained with the
reference load unchanged.

`num_mcts_searches > 0` runs the device tree search of mcts.py.  `learn()` runs PPO over collector.RolloutCollector or AlphaZero
self-play over the device tree search (ppo.py), chosen by `algorithm_cls` like the reference does.
"""
from __future__ import annotations

import json

import torch

from .search import BasicPolicy, RolloutSearch, check_tensor_core_search, chunk_plan
from .specs import SynthSpec

_ENV_KINDS = {"PermutationEnv": 0, "LinearFunctionEnv": 1, "CliffordEnv": 2, "PauliNetworkEnv": 3}


def gate_list_to_circuit(gate_list, num_qubits=None):
    """rl/synthesis.py:141-147 (needs Qiskit)."""
    if num_qubits is None:
        num_qubits = max(max(gate_args) for _, gate_args in gate_list) + 1
    from .wire import gates_to_circuit
    return gates_to_circuit(gate_list, num_qubits)


class RLSynthesis:
    def __init__(self, env, rl_config: dict | None, model_config: dict | None, model_path: str | None = None, device=None,
                 policy_cls: str = "twisterl.nn.BasicPolicy", algorithm_cls: str = "twisterl.rl.PPO"):
        self.env = env
        self.env_config = env.to_json()
        # config objects (configs.PPOConfig / AlphaZeroConfig / BasicPolicyConfig, as in the reference) or dicts in their JSON schema
        if hasattr(rl_config, "to_json"):
            algorithm_cls, rl_config = rl_config.algorithm_cls, rl_config.to_json()
        if hasattr(model_config, "to_json"):
            policy_cls, model_config = model_config.policy_cls, model_config.to_json()
        self.rl_config = dict(rl_config or {})
        self.model_config = dict(model_config or {})
        self.policy_cls = policy_cls
        self.algorithm_cls = algorithm_cls
        if policy_cls.split(".")[-1] != "BasicPolicy":
            raise NotImplementedError(f"policy class {policy_cls} is not supported (BasicPolicy only)")
        self.device = device
        self.policy = self._init_policy(model_path)
        self._searches = {}

    # ---- construction ---------------------------------------------------------------------------------
    @classmethod
    def from_config_json(cls, config_path, model_path=None, device=None):
        """rl/synthesis.py:54-77: `{env_cls, env, policy_cls, policy, algorithm_cls, algorithm}`."""
        full = json.load(open(config_path))
        env = SynthSpec.from_json(full["env_cls"], full["env"])      # Qiskit-free problem spec (specs.py); a reference *Gym object works too
        return cls(env, full.get("algorithm"), full.get("policy"), model_path, device=device,
                   policy_cls=full.get("policy_cls", "twisterl.nn.BasicPolicy"), algorithm_cls=full.get("algorithm_cls", "twisterl.rl.PPO"))

    def _init_policy(self, model_path):
        """rl/synthesis.py:95-110: policy(obs_shape, num_actions, **model_config); checkpoint = plain state_dict."""
        mc = self.model_config
        pol = BasicPolicy(self.env.obs_shape(), self.env.num_actions(), embedding_size=mc.get("embedding_size", 512),
                          common_layers=tuple(mc.get("common_layers", (256,))), policy_layers=tuple(mc.get("policy_layers", ())),
                          value_layers=tuple(mc.get("value_layers", ())))
        if model_path is not None:
            pol.load_state_dict(torch.load(model_path, map_location="cpu", weights_only=True))
        return pol.eval()

    def to_json(self):
        return {"env_cls": f"qiskit_gym.envs.synthesis.{self.env.cls_name}", "env": self.env_config, "policy_cls": self.policy_cls,
                "policy": self.model_config, "algorithm_cls": self.algorithm_cls, "algorithm": self.rl_config}

    def save(self, config_path, model_path=None):
        with open(config_path, "w") as f:
            json.dump(self.to_json(), f, indent=2)
        if model_path is not None:
            with open(model_path, "wb") as f:
                torch.save(self.policy.state_dict(), f)

    # ---- synthesis ------------------------------------------------------------------------------------
    def _env_args(self, **override):
        """(env kind, num_qubits, gateset, the env config's other entries updated with `override`): what a device engine is built from."""
        cfg = self.env_config
        kw = {k: v for k, v in cfg.items() if k not in ("num_qubits", "gateset")}
        return _ENV_KINDS[self.env.cls_name], cfg["num_qubits"], cfg["gateset"], {**kw, **override}

    def _search(self, num_searches: int, targets_per_launch: int | None = None, matmul_precision: str = "f32") -> RolloutSearch:
        """The cached search of `num_searches` rollouts per target: the single-target one, or with targets_per_launch the one solve_many
        uses (rebuilt only when a call needs more targets per launch than it holds).  matmul_precision="tensor_core": the "tensor_core"
        backend, cached under its own key (it never replaces the f32 search) and with no fall-back.  A search refreshes its policy handle
        from self.policy itself, so a weight update does not rebuild it."""
        key = num_searches if targets_per_launch is None else ("many", num_searches)
        if matmul_precision == "tensor_core":
            key = ("tensor_core", key)
        rs = self._searches.get(key)
        if rs is not None and targets_per_launch is not None and rs.targets_per_launch < targets_per_launch:
            rs = None
        if rs is None:
            self._searches.pop(key, None)                # (frees the old engine before the new one allocates)
            kind, n, gs, kw = self._env_args(add_perms=False)

            def make(backend):
                return RolloutSearch(kind, n, gs, self.policy, num_searches, device=self.device, policy_backend=backend,
                                     targets_per_launch=targets_per_launch or 1, **kw)
            if matmul_precision == "tensor_core":
                rs = make("tensor_core")
            else:
                try:
                    rs = make("persistent")
                    rs.check_supported()
                except NotImplementedError:
                    # outside the one-launch search's limits (Permutation wider than 64 qubits, a layer wider than 1024, policy + env larger
                    # than one SM's shared memory): the PyTorch policy on dense observations has none of them
                    rs = make("torch")
            self._searches[key] = rs
        return rs

    def _mcts(self, num_searches: int, num_mcts_searches: int, C: float, reuse_tree: bool = False):
        from .mcts import MCTSSearch
        key = ("mcts", num_searches, num_mcts_searches, C, reuse_tree)
        ms = self._searches.get(key)
        if ms is None:
            kind, n, gs, kw = self._env_args(add_perms=False)
            ms = MCTSSearch(kind, n, gs, self.policy, num_searches, num_mcts_searches, C=C, device=self.device, reuse_tree=reuse_tree, **kw)
            self._searches[key] = ms
        return ms

    def solve(self, state, deterministic: bool = False, num_searches: int = 100, num_mcts_searches: int = 0, C: float = 2 ** 0.5,
              max_expand_depth: int = 1, seed: int = 0, reuse_tree: bool = False):
        """twisterl `Algorithm.solve`: the action list of the best successful rollout, or None.
        reuse_tree (tree search only): every decision but the first starts from the subtree below the action played (mcts.MCTSSearch)."""
        if reuse_tree and not num_mcts_searches:
            raise ValueError("reuse_tree needs a tree search (num_mcts_searches > 0)")
        if num_mcts_searches:
            if max_expand_depth != 1:
                raise NotImplementedError("max_expand_depth != 1 is not supported by the device tree search (mcts.py)")
            return self._mcts(int(num_searches), int(num_mcts_searches), float(C), bool(reuse_tree)).solve(state, deterministic=deterministic,
                                                                                                             seed=seed).actions
        return self._search(int(num_searches)).solve(state, deterministic=deterministic, seed=seed).actions

    def solve_many(self, states, deterministic: bool = False, num_searches: int = 100, num_mcts_searches: int = 0, seed: int = 0,
                   max_rollouts: int = 65536, matmul_precision: str = "f32"):
        """`solve` for many targets in few launches: a list with, for each state, the action list of its best successful rollout or None.
        Target t's result is that of solve(states[t]) on rollout ids t*num_searches .. (t+1)*num_searches - 1 (search.RolloutSearch.solve_many),
        so solve_many([x])[0] == solve(x).  Up to max_rollouts rollouts run per launch (the one-launch search keeps ~4 KB of first-layer
        accumulators per rollout at the default network: 65 536 rollouts ~ 256 MB).
        matmul_precision: "f32" (the default: the searches of solve) or "tensor_core" (RolloutSearch's "tensor_core" backend: the policy on
        tcgen05 tensor cores, for large launches).  The two round differently, so "tensor_core" results equal a single-target "tensor_core"
        search, not solve(); it raises NotImplementedError where it cannot run (more than 127 actions, a Permutation wider than 64 qubits, a
        device that is not sm_100) instead of falling back to another arithmetic."""
        if num_mcts_searches:
            raise NotImplementedError("solve_many runs rollout searches only (num_mcts_searches = 0): use solve() for the tree search")
        if matmul_precision not in ("f32", "tensor_core"):
            raise ValueError(f"matmul_precision must be f32 or tensor_core (got {matmul_precision!r})")
        states = list(states)
        num_searches = int(num_searches)
        if num_searches < 1:
            raise ValueError("num_searches must be >= 1")
        chunk_plan(len(states), 1, num_searches)         # ValueError for targets x rollouts >= 2^30, before anything is allocated
        if matmul_precision == "tensor_core":
            check_tensor_core_search(_ENV_KINDS[self.env.cls_name], self.env_config["num_qubits"], self.env.num_actions(), self.device)
        if not states:
            return []
        tpl = min(len(states), max(1, int(max_rollouts) // num_searches))
        res = self._search(num_searches, tpl, matmul_precision).solve_many(states, deterministic=deterministic, seed=seed)
        return [r.actions for r in res]

    def synth_many(self, inputs, deterministic: bool = False, num_searches: int = 100, num_mcts_searches: int = 0, seed: int = 0,
                   max_rollouts: int = 65536, matmul_precision: str = "f32"):
        """`synth` for many inputs (solve_many): a list of circuits (or gate lists), None where a target has no successful rollout."""
        inputs = list(inputs)
        actions = self.solve_many([self.env.get_state(x) for x in inputs], deterministic, num_searches, num_mcts_searches, seed, max_rollouts,
                                  matmul_precision)
        out = []
        for x, a in zip(inputs, actions):
            if a is None:
                out.append(None)
                continue
            self.env.get_state(x)                        # the env object's per-target state (PauliNetwork rotation parameters), as synth leaves it
            out.append(self.env.build_circuit_from_solution(a, x))
        return out

    def synth(self, input, deterministic: bool = False, num_searches: int = 100, num_mcts_searches: int = 0, C: float = 2 ** 0.5,
              max_expand_depth: int = 1, seed: int = 0, reuse_tree: bool = False):
        """rl/synthesis.py:112-126.  Returns the synthesised circuit (QuantumCircuit with Qiskit, else a gate list) or None."""
        state = self.env.get_state(input)
        actions = self.solve(state, deterministic, num_searches, num_mcts_searches, C, max_expand_depth, seed=seed, reuse_tree=reuse_tree)
        if actions is not None:
            return self.env.build_circuit_from_solution(actions, input)

    def learn(self, initial_difficulty=1, num_iterations=int(1e10), tb_path=None, log=None, seed: int = 0, matmul_precision: str = "f32",
              update_precision: str = "f32"):
        """rl/synthesis.py:128-139: PPO (`twisterl.rl.PPO`) or AlphaZero (`twisterl.rl.AZ`) on the device (ppo.py).  The trained
        policy is `self.policy` (searches built before the call are dropped so that `synth` uses the new weights).
        matmul_precision (PPO): how the collector runs the policy — "f32" (the reference's arithmetic, the default), "tf32", "bf16", or
        "tensor_core" (packed observations and the tcgen05 policy: RolloutCollector.collect_packed).
        update_precision (PPO): "f32" (the default) or "tensor_core" (the update's forward and backward on the tcgen05 kernels; needs
        matmul_precision="tensor_core")."""
        from . import ppo
        algo = self.algorithm_cls.split(".")[-1]
        if algo not in ("PPO", "AZ"):
            raise NotImplementedError(f"algorithm class {self.algorithm_cls} is not supported (twisterl.rl.PPO, twisterl.rl.AZ)")
        if algo == "AZ" and matmul_precision != "f32":
            raise NotImplementedError("matmul_precision applies to PPO only (AlphaZero evaluates its policy inside the tree search)")
        if algo == "AZ" and update_precision != "f32":
            raise NotImplementedError("update_precision applies to PPO only (the AlphaZero update runs in f32 PyTorch)")
        kind, n, gs, kw = self._env_args()
        if algo == "PPO":
            kw["matmul_precision"] = matmul_precision
            kw["update_precision"] = update_precision
        trainer = (ppo.PPO if algo == "PPO" else ppo.AlphaZero)(kind, n, gs, self.policy, self.rl_config, device=self.device, seed=seed, **kw)
        if hasattr(self.env, "difficulty"):
            self.env.difficulty = initial_difficulty                # rl/synthesis.py:129 (a reference *Gym object; a SynthSpec owns no env)
        try:
            return trainer.learn(initial_difficulty=initial_difficulty, num_iterations=num_iterations, tb_path=tb_path, log=log)
        except KeyboardInterrupt:
            # rl/synthesis.py:137-139: stopping a run by hand keeps the policy trained so far (metrics.jsonl under tb_path holds the history)
            return getattr(trainer, "history", None)
        finally:
            self.policy = trainer.policy.eval()
            self._searches = {}
