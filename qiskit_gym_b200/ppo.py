"""PPO over the on-device collector — what `RLSynthesis.learn()` runs (reference src/qiskit_gym/rl/synthesis.py:128-139
-> twisterl `PPO.learn`; hyper-parameters and their JSON schema from src/qiskit_gym/rl/configs.py:72-240).

The reference hands the env to twisterl, whose Rust collectors step `num_episodes` cloned envs on a rayon pool and whose
Python side runs the clipped-surrogate update.  Here the collection is `collector.RolloutCollector` (every env of one
`BatchedEnv` plays episodes back to back on the GPU, GAE on the device) and the update is plain PyTorch on the tensors
the collector left on the device; nothing crosses the PCIe bus during training except the logged scalars.  Under `torch.distributed` (one process per GPU) every
rank collects on its own environments and the gradients are averaged with one all-reduce per optimiser step (`sync_gradients`).

Config: the nested dict `PPOConfig.to_json()` writes (configs.py:205-240) —
    collecting {num_cores (ignored: the batch is the parallelism), num_episodes, lambda, gamma}
    training   {num_epochs, vf_coef, ent_coef, clip_ratio, normalize_advantage}
    learning   {diff_threshold, diff_max, diff_metric}      optimizer {lr}
    evals      {name: {num_episodes, deterministic, num_searches, num_mcts_searches, num_cores, C}}
    logging    {log_freq, checkpoint_freq}
Missing keys take the reference's defaults.  twisterl itself is not in the reference tree, so the loop below follows its
documented semantics (configs.py docstrings), not its code: one iteration = collect >= num_episodes episodes at the current
difficulty, `num_epochs` full-batch updates, evaluate, and raise the difficulty by one when `evals[diff_metric]` reaches
`diff_threshold` (up to `diff_max`).
"""
from __future__ import annotations

import json
import os
import time

import torch

from .collector import RolloutCollector, decision_seed, unpack_bits
from .engine import BatchedEnv

_EVAL_DEFAULT = {"num_episodes": 100, "deterministic": True, "num_searches": 1, "num_mcts_searches": 0, "num_cores": 32, "C": 1.41}
# AlphaZeroConfig (configs.py:325-360)
_AZ_DEFAULTS = {
    "collecting": {"num_cores": 32, "num_episodes": 128, "num_mcts_searches": 1000, "C": 1.41, "max_expand_depth": 1},
    "training": {"num_epochs": 10},
    "learning": {"diff_threshold": 0.85, "diff_max": 256, "diff_metric": "mcts_100"},
    "optimizer": {"lr": 3e-4},
    "evals": {"ppo_deterministic": dict(_EVAL_DEFAULT), "ppo_10": dict(_EVAL_DEFAULT, deterministic=False, num_searches=10),
              "mcts_100": dict(_EVAL_DEFAULT, num_mcts_searches=100)},
    "logging": {"log_freq": 1, "checkpoint_freq": 10},
}
_DEFAULTS = {
    "collecting": {"num_cores": 32, "num_episodes": 1024, "lambda": 0.995, "gamma": 0.995},
    "training": {"num_epochs": 10, "vf_coef": 0.8, "ent_coef": 0.01, "clip_ratio": 0.1, "normalize_advantage": False},
    "learning": {"diff_threshold": 0.85, "diff_max": 256, "diff_metric": "ppo_deterministic"},
    "optimizer": {"lr": 3e-4},
    "evals": {"ppo_deterministic": {"num_episodes": 100, "deterministic": True, "num_searches": 1, "num_mcts_searches": 0, "num_cores": 32, "C": 1.41},
              "ppo_10": {"num_episodes": 100, "deterministic": False, "num_searches": 10, "num_mcts_searches": 0, "num_cores": 32, "C": 1.41}},
    "logging": {"log_freq": 1, "checkpoint_freq": 10},
}


def merged_config(cfg: dict | None, algorithm: str = "PPO") -> dict:
    """The reference's defaults (PPOConfig configs.py:133-166, AlphaZeroConfig 325-360) overlaid with `cfg`; validates like
    `PPOConfig.validate` / `AlphaZeroConfig.validate` (168-196, 364-391)."""
    base = _AZ_DEFAULTS if algorithm == "AZ" else _DEFAULTS
    out = {k: dict(v) for k, v in base.items()}
    out["evals"] = {k: dict(v) for k, v in base["evals"].items()}
    for sec, val in (cfg or {}).items():
        if sec == "evals":
            out["evals"] = {name: {**_EVAL_DEFAULT, **dict(ev)} for name, ev in dict(val).items()}
        elif sec in out:
            out[sec].update(dict(val))
    c, t, l = out["collecting"], out["training"], out["learning"]
    if c["num_episodes"] <= 0:
        raise ValueError("num_episodes must be > 0")
    if algorithm == "AZ":
        if c["num_mcts_searches"] <= 0:
            raise ValueError("num_mcts_searches must be > 0")
        if c["C"] <= 0:
            raise ValueError("C must be > 0")
        if c["max_expand_depth"] < 1:
            raise ValueError("max_expand_depth must be >= 1")
    else:
        if not 0.0 <= c["lambda"] <= 1.0:
            raise ValueError("gae_lambda must be in [0, 1]")
        if not 0.0 <= c["gamma"] <= 1.0:
            raise ValueError("gamma must be in [0, 1]")
        if t["clip_ratio"] <= 0:
            raise ValueError("clip_ratio must be > 0")
    if t["num_epochs"] <= 0:
        raise ValueError("num_epochs must be > 0")
    if not 0.0 <= l["diff_threshold"] <= 1.0:
        raise ValueError("diff_threshold must be in [0, 1]")
    if l["diff_max"] < 1:
        raise ValueError("diff_max must be >= 1")
    if l["diff_metric"] not in out["evals"]:
        raise ValueError(f"diff_metric '{l['diff_metric']}' not found in evals: {list(out['evals'])}")
    for name, ev in out["evals"].items():
        if ev["num_episodes"] <= 0 or ev["num_searches"] <= 0 or ev["num_mcts_searches"] < 0 or ev["C"] <= 0:
            raise ValueError(f"Invalid eval '{name}'")
    return out


# ---- data-parallel training: one process per GPU, every rank collects on its own shard of environments, gradients averaged ----
def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) else None


def sync_gradients(params, group=None) -> None:
    """Average the gradients over the ranks with ONE all-reduce of the flattened gradient (NCCL on GPUs, gloo in the CPU tests)."""
    dist = _dist()
    if dist is None:
        return
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= dist.get_world_size(group)
    o = 0
    for g in grads:
        g.copy_(flat[o:o + g.numel()].view_as(g))
        o += g.numel()


def broadcast_parameters(module: torch.nn.Module, src: int = 0, group=None) -> None:
    """Every replica starts from rank `src`'s weights."""
    dist = _dist()
    if dist is None:
        return
    for t in list(module.parameters()) + list(module.buffers()):
        dist.broadcast(t.data, src=src, group=group)


def agree_min(value: int, device=None, group=None) -> int:
    """The smallest `value` over the ranks (how many optimiser steps an epoch makes: every rank must make the same number)."""
    dist = _dist()
    if dist is None:
        return int(value)
    t = torch.tensor([int(value)], dtype=torch.int64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return int(t.item())


def mean_over_ranks(value: float, device=None, group=None) -> float:
    dist = _dist()
    if dist is None:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return float(t.item()) / dist.get_world_size(group)


class Trainer:
    """What PPO and AlphaZero share: the envs, the difficulty curriculum, the evals, logging and checkpoints.
    Subclasses provide `iterate() -> dict` (collect + update, returns the iteration's scalars)."""

    algorithm = "PPO"

    def __init__(self, env_kind: int, num_qubits: int, gateset, policy: torch.nn.Module, config: dict | None = None, device=None,
                 seed: int = 0, minibatch_size: int | None = None, **env_kwargs):
        self.cfg = merged_config(config, self.algorithm)
        self.spec = (env_kind, num_qubits, list(gateset), dict(env_kwargs))
        self.seed = int(seed)
        self.minibatch_size = minibatch_size
        self._eval_envs = {}
        self._eval_mcts = {}
        self.iteration = 0
        self.history = []
        self._difficulty = int(env_kwargs.get("difficulty", 1))
        self.env = self._make_env(int(self.cfg["collecting"]["num_episodes"]), device)
        self.device = self.env.device
        self.policy = policy.to(self.device)
        d = _dist()
        self.rank, self.world = (d.get_rank(), d.get_world_size()) if d else (0, 1)
        broadcast_parameters(self.policy)
        self.opt = torch.optim.Adam(self.policy.parameters(), lr=float(self.cfg["optimizer"]["lr"]))

    def _make_env(self, batch: int, device) -> BatchedEnv:
        kind, n, gs, kw = self.spec
        return BatchedEnv(kind, n, gs, batch, device=device, **kw)

    # ---- difficulty (Env::set_difficulty on every env the trainer owns) -------------------------------------------
    @property
    def difficulty(self) -> int:
        return self._difficulty

    @difficulty.setter
    def difficulty(self, d: int):
        self._difficulty = int(d)
        self.env.difficulty = int(d)

    def _episode_steps(self) -> int:
        """An episode lasts at most depth = min(depth_slope * difficulty, max_depth) decisions (e.g. clifford.rs:306-319)."""
        c = self.env.cfg
        return int(max(1, min(int(c.depth_slope) * self.difficulty, int(c.max_depth))))

    def _minibatches(self, n: int):
        """Index sets of one epoch.  Under torch.distributed every rank makes the same number of optimiser steps (the smallest count
        any rank would make), each over an equal share of its own samples."""
        mb = n if not self.minibatch_size else min(int(self.minibatch_size), n)
        steps = agree_min(max(1, -(-n // max(mb, 1))), self.device)
        mb = -(-n // steps)
        perm = torch.randperm(n, device=self.device) if steps > 1 else None
        for k in range(steps):
            yield slice(k * mb, (k + 1) * mb) if perm is None else perm[k * mb:(k + 1) * mb]

    def _step(self, loss):
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        sync_gradients(list(self.policy.parameters()))
        self.opt.step()

    def _probs(self, obs):
        with torch.no_grad():
            logits, _ = self.policy(obs)
            return torch.softmax(logits.float(), dim=-1).contiguous()

    # ---- evaluation ----------------------------------------------------------------------------------------------------
    def evaluate(self, name: str) -> float:
        """Success rate of `evals[name]`: num_episodes fresh targets at the current difficulty, each tried with `num_searches`
        rollouts (greedy or sampled; with a tree search of `num_mcts_searches` simulations per decision when that is > 0); an
        episode counts when any of its rollouts ends in success (configs.py:25-35)."""
        ev = self.cfg["evals"][name]
        E, sims = int(ev["num_episodes"]), int(ev.get("num_mcts_searches", 0))
        base = decision_seed(self.seed ^ 0x5EED5EED, 1_000_003 * (self.iteration + 1) + 7919 * self.rank)
        steps = self._episode_steps()
        self.policy.eval()
        if sims:
            from .mcts import MCTSSearch
            key = (E, sims, float(ev["C"]))
            ms = self._eval_mcts.get(key)
            if ms is None:
                kind, n, gs, kw = self.spec
                ms = MCTSSearch(kind, n, gs, self.policy, E, sims, C=float(ev["C"]), device=self.device.index, **kw)
                self._eval_mcts[key] = ms
            ms.policy = self.policy
            env = ms.env
        else:
            env = self._eval_envs.get(E)
            if env is None:
                env = self._eval_envs[E] = self._make_env(E, self.device.index)
        env.difficulty = self.difficulty
        env.reset(seed=base)
        env.snapshot()
        solved = torch.zeros(E, dtype=torch.bool, device=self.device)
        for s in range(int(ev["num_searches"])):
            if s:
                env.restore()
            for k in range(steps):
                weights = ms.decide(k) if sims else self._probs(env.observe())
                env.collect_step(weights, decision_seed(base, (s + 1) * 4099 + k), deterministic=bool(ev["deterministic"]), obs=False)
            solved |= env.status()[2]
        return mean_over_ranks(float(solved.float().mean().item()), self.device)

    def iterate(self) -> dict:
        raise NotImplementedError

    # ---- the loop ------------------------------------------------------------------------------------------------------
    def learn(self, initial_difficulty: int = 1, num_iterations: int = int(1e10), tb_path: str | None = None, log=None, stop_at_max: bool = False):
        """rl/synthesis.py:128-139.  Returns the history (one dict per iteration).  `tb_path`: directory for `metrics.jsonl` and
        checkpoints (`checkpoint_<iteration>.pt`, a plain state_dict like the reference's examples/models)."""
        L, lg = self.cfg["learning"], self.cfg["logging"]
        self.difficulty = int(initial_difficulty)
        fh = None
        if tb_path and self.rank == 0:
            os.makedirs(tb_path, exist_ok=True)
            fh = open(os.path.join(tb_path, "metrics.jsonl"), "a")
        try:
            for _ in range(int(num_iterations)):
                t0 = time.time()
                rec = {"iteration": self.iteration, "difficulty": self.difficulty}
                rec.update(self.iterate())
                if self.iteration % max(1, int(lg["log_freq"])) == 0:
                    for name in self.cfg["evals"]:
                        rec[f"eval/{name}"] = self.evaluate(name)
                    metric = rec[f"eval/{L['diff_metric']}"]
                    if metric >= float(L["diff_threshold"]) and self.difficulty < int(L["diff_max"]):
                        self.difficulty = self.difficulty + 1
                rec["seconds"] = time.time() - t0
                self.history.append(rec)
                if fh:
                    fh.write(json.dumps(rec) + "\n")
                    fh.flush()
                    if (self.iteration + 1) % max(1, int(lg["checkpoint_freq"])) == 0:
                        torch.save(self.policy.state_dict(), os.path.join(tb_path, f"checkpoint_{self.iteration + 1}.pt"))
                if log:
                    log(rec)
                self.iteration += 1
                if stop_at_max and self.difficulty >= int(L["diff_max"]) and rec.get(f"eval/{L['diff_metric']}", 0.0) >= float(L["diff_threshold"]):
                    break
        finally:
            if fh:
                fh.close()
        return self.history


class PPO(Trainer):
    """`PPO(env kind, num_qubits, gateset, policy, config, **BatchedEnv keyword arguments).learn(...)`."""

    algorithm = "PPO"

    def __init__(self, env_kind: int, num_qubits: int, gateset, policy: torch.nn.Module, config: dict | None = None, device=None,
                 seed: int = 0, use_twists: bool = True, minibatch_size: int | None = None, matmul_precision: str = "f32",
                 update_precision: str = "f32", **env_kwargs):
        """matmul_precision: "f32" (default), "tf32" or "bf16" run the policy in PyTorch on dense observations (RolloutCollector.collect);
        "tensor_core" collects with packed-bit observations and the tcgen05 policy (RolloutCollector.collect_packed, twists included) and
        the update unpacks each minibatch's observations from the bits.  "tensor_core" raises NotImplementedError where that path cannot run
        (more than 127 actions, a value head that is not one Linear, a device that is not sm_100).
        update_precision: "f32" (default) runs the update's forward and backward in PyTorch; "tensor_core" runs them on the tcgen05 kernels
        (TensorCorePolicy.forward_train) from the packed rollout's bits, so it needs matmul_precision="tensor_core".  The loss is the same code."""
        if matmul_precision not in ("f32", "tf32", "bf16", "tensor_core"):
            raise ValueError(f"matmul_precision must be one of f32, tf32, bf16, tensor_core (got {matmul_precision!r})")
        if update_precision not in ("f32", "tensor_core"):
            raise ValueError(f"update_precision must be f32 or tensor_core (got {update_precision!r})")
        if update_precision == "tensor_core" and matmul_precision != "tensor_core":
            raise ValueError('update_precision="tensor_core" trains on the packed rollout\'s bits: it needs matmul_precision="tensor_core"')
        super().__init__(env_kind, num_qubits, gateset, policy, config, device=device, seed=seed, minibatch_size=minibatch_size, **env_kwargs)
        self.tensor_core = matmul_precision == "tensor_core"
        self.collector = RolloutCollector(self.env, self.policy, gamma=self.cfg["collecting"]["gamma"], lam=self.cfg["collecting"]["lambda"],
                                          use_twists=use_twists, seed=seed + 104729 * self.rank, first_env_id=self.rank * self.env.batch,
                                          matmul_precision="f32" if self.tensor_core else matmul_precision)
        if self.tensor_core:
            self.collector.tensor_core_policy()          # fails here, not in the first iteration, where the tensor-core policy cannot run
        self.update_tc = update_precision == "tensor_core"
        self._train_tcp = None

    def iterate(self) -> dict:
        steps = self._episode_steps()
        ro = self.collector.collect_packed(steps) if self.tensor_core else self.collector.collect(steps)
        episodes, success = ro.episode_stats()
        rec = {"episodes": episodes, "collect_success": success,
               "mean_reward": float(ro.rewards[ro.valid].mean().item()) if bool(ro.valid.any()) else 0.0}
        rec.update(self.update(ro))
        return rec

    def update(self, ro) -> dict:
        """`num_epochs` passes of the clipped-surrogate update over the valid decisions of a Rollout."""
        t = self.cfg["training"]
        idx = ro.valid.reshape(-1).nonzero(as_tuple=False).squeeze(1)
        if ro.obs is None:          # packed rollout: keep the gathered bits (32x smaller) and unpack one minibatch at a time
            bits = ro.obs_bits.reshape(-1, ro.obs_bits.shape[-1])[idx]
            shape = tuple(self.env.obs_shape())
            obs_of = lambda sel: unpack_bits(bits[sel], ro.obs_size).reshape((-1,) + shape)      # noqa: E731
        else:
            obs = ro.obs.reshape((-1,) + tuple(ro.obs.shape[2:]))[idx]
            obs_of = lambda sel: obs[sel]                                                         # noqa: E731
        forward = (lambda sel: self._train_policy(int(bits[sel].shape[0])).forward_train(self.policy, bits[sel])) if self.update_tc \
            else (lambda sel: self.policy(obs_of(sel)))                                           # noqa: E731
        act = ro.policy_actions.reshape(-1)[idx]
        logp_old = ro.logp.reshape(-1)[idx]
        adv = ro.advantages.reshape(-1)[idx]
        ret = ro.returns.reshape(-1)[idx]
        if t["normalize_advantage"] and adv.numel() > 1:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        n = int(idx.numel())
        clip = float(t["clip_ratio"])
        self.policy.train()
        stats = {}
        for _ in range(int(t["num_epochs"])):
            for sel in self._minibatches(n):
                logits, value = forward(sel)
                logp_all = torch.log_softmax(logits.float(), dim=-1)
                logp = logp_all.gather(1, act[sel][:, None]).squeeze(1)
                ratio = torch.exp(logp - logp_old[sel])
                a = adv[sel]
                pi_loss = -torch.min(ratio * a, torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * a).mean()
                v_loss = torch.nn.functional.mse_loss(value.float().reshape(-1), ret[sel])
                entropy = -(logp_all.exp() * logp_all).sum(-1).mean()
                loss = pi_loss + float(t["vf_coef"]) * v_loss - float(t["ent_coef"]) * entropy
                self._step(loss)
                stats = {"loss": loss.detach(), "pi_loss": pi_loss.detach(), "v_loss": v_loss.detach(), "entropy": entropy.detach(),
                         "clip_frac": ((ratio - 1.0).abs() > clip).float().mean().detach()}
        self.policy.eval()
        return {k: float(v.item()) for k, v in stats.items()} | {"samples": n}

    def _train_policy(self, rows: int):
        """The update's training handle (TensorCorePolicy with the backward pass), grown geometrically when a minibatch outgrows it."""
        from .policy import TensorCorePolicy
        tcp = self._train_tcp
        if tcp is None or tcp.max_batch < rows:
            cap = max(rows, 2 * tcp.max_batch) if tcp is not None else rows
            tcp = self._train_tcp = TensorCorePolicy(self.policy, max_batch=cap, device=self.device, with_value=True, training=True)
        return tcp


class AlphaZero(Trainer):
    """Self-play with the device tree search (mcts.py) and the AlphaZero update: every decision of every episode runs
    `num_mcts_searches` PUCT simulations; the action is sampled from the root's visit counts; the policy is trained towards
    the visit distribution (cross entropy) and the value head towards the episode's return-to-go (undiscounted, like the tree's
    own back-up; episodes cut by the end of the collection bootstrap from the value head).  Config: AlphaZeroConfig.to_json()
    (configs.py:404-429).  twisterl's AZ is not in the reference tree: this follows the config docstrings (295-323), not its code.
    use_twists: self-play runs the twisted tree search (MCTSSearch(use_twists=True)), so the policy learns in the env's symmetry frames
    as PPO's collector trains it.  A sample is the root observation as the root evaluation saw it (in frame k), and its target is the
    visit distribution in the policy's action order, tgt[act_perm[k][a]] = w[a]; the env still plays the sampled env action.  Raises
    before anything is allocated where the twisted tree search cannot run (mcts.check_twisted_tree_search).
    matmul_precision: how self-play's tree search evaluates the policy, "f32" (the default: the fused FFMA kernel, or the PyTorch module
    where that cannot run) or "tensor_core" (MCTSSearch(policy_backend="tensor_core"): the tcgen05 policy, for thousands of episodes per
    iteration; NotImplementedError, before anything is allocated, where it cannot run).  The evals, the bootstrap value and the update
    stay f32 PyTorch either way."""

    algorithm = "AZ"

    def __init__(self, env_kind: int, num_qubits: int, gateset, policy: torch.nn.Module, config: dict | None = None, device=None,
                 seed: int = 0, minibatch_size: int | None = None, vf_coef: float = 1.0, use_twists: bool = False, matmul_precision: str = "f32",
                 **env_kwargs):
        from .mcts import MCTSSearch, check_tensor_core_tree_search, check_twisted_tree_search
        if matmul_precision not in ("f32", "tensor_core"):
            raise ValueError(f"AlphaZero's matmul_precision must be f32 or tensor_core (got {matmul_precision!r})")
        self.use_twists = bool(use_twists)
        self.policy_backend = "tensor_core" if matmul_precision == "tensor_core" else "auto"
        if self.use_twists:
            check_twisted_tree_search(env_kind, num_qubits, policy, self.policy_backend, env_kwargs)
        if matmul_precision == "tensor_core":
            check_tensor_core_tree_search(env_kind, num_qubits, len(gateset), policy, device)
        self._mcts_cls = MCTSSearch
        self._policy_for_env = policy
        self.vf_coef = float(vf_coef)
        super().__init__(env_kind, num_qubits, gateset, policy, config, device=device, seed=seed, minibatch_size=minibatch_size, **env_kwargs)
        self.counter = 0

    def _make_env(self, batch: int, device) -> BatchedEnv:
        if hasattr(self, "env"):                       # eval envs without a tree search
            return super()._make_env(batch, device)
        c = self.cfg["collecting"]
        if int(c["max_expand_depth"]) != 1:
            raise NotImplementedError("max_expand_depth != 1 is not supported by the device tree search (mcts.py)")
        kind, n, gs, kw = self.spec
        twist_kw = {"use_twists": True} if self.use_twists else {}
        self.search = self._mcts_cls(kind, n, gs, self._policy_for_env, batch, int(c["num_mcts_searches"]), C=float(c["C"]), device=device,
                                     policy_backend=self.policy_backend, **twist_kw, **kw)
        return self.search.env

    def iterate(self) -> dict:
        rec, obs, tgt_pi, tgt_v, _ = self.self_play()
        n = int(obs.shape[0])
        self.policy.train()
        stats = {}
        for _ in range(int(self.cfg["training"]["num_epochs"])):
            for sel in self._minibatches(n):
                logits, value = self.policy(obs[sel])
                logp_all = torch.log_softmax(logits.float(), dim=-1)
                pi_loss = -(tgt_pi[sel] * logp_all).sum(-1).mean()
                v_loss = torch.nn.functional.mse_loss(value.float().reshape(-1), tgt_v[sel])
                loss = pi_loss + self.vf_coef * v_loss
                self._step(loss)
                stats = {"loss": loss.detach(), "pi_loss": pi_loss.detach(), "v_loss": v_loss.detach()}
        self.policy.eval()
        rec.update({k: float(v.item()) for k, v in stats.items()} | {"samples": n})
        return rec

    def self_play(self):
        """One collection of self-play: -> (episode stats, the training samples' observations, policy targets and value targets, and
        the samples' indices into the flattened [steps, envs] decisions)."""
        from .collector import gae
        env, ms, T, B = self.env, self.search, self._episode_steps(), self.env.batch
        ms.policy = self.policy.eval()
        dev, A = self.device, env.num_actions()
        obs_buf = torch.empty((T, B) + tuple(env.obs_shape()), dtype=torch.float32, device=dev)
        pi = torch.zeros((T, B, A), dtype=torch.float32, device=dev)
        actions = torch.full((T, B), -1, dtype=torch.int32, device=dev)
        rewards = torch.zeros((T, B), dtype=torch.float32, device=dev)
        dones = torch.zeros((T, B), dtype=torch.bool, device=dev)
        succ = torch.zeros((T, B), dtype=torch.bool, device=dev)
        for t in range(T):
            s = decision_seed(self.seed + 104729 * self.rank, self.counter)
            env.reset_select(s, self.rank * B)
            if self.use_twists:
                env.search_begin(s, self.rank * B)   # the frames' seed and global ids (AZ reads no search returns)
            w = ms.decide(t)                         # grows the trees from the root observation, leaves N(a) / sum N in ms.weights
            if ms.backend != "torch":
                # the packed backends observe into bits only (ms.root_bits): the training sample is what the root evaluation saw
                # (for PauliNetwork with add_perms that includes the qubit permutation observe() picked)
                obs_buf[t].copy_(unpack_bits(ms.root_bits, env._obs_size).reshape(obs_buf[t].shape))
            else:
                obs_buf[t].copy_(env.obs)
            if self.use_twists:
                pi[t].scatter_(1, ms.act_table[ms.root_twist.long()].long(), w)      # the target in the policy's action order
            else:
                pi[t].copy_(w)
            env.collect_step(w, s, deterministic=False, obs=False, chosen=actions[t], reward=rewards[t], done=dones[t], success=succ[t])
            self.counter += 1
        valid = actions >= 0
        values = torch.zeros((T + 1, B), dtype=torch.float32, device=dev)
        with torch.no_grad():
            values[T] = self.policy(env.observe())[1].float().reshape(-1)
        _, ret = gae(rewards, values, dones, 1.0, 1.0, valid)        # V = 0 inside, gamma = lambda = 1: the return-to-go (+ bootstrap)
        fin = dones & valid
        n_ep = int(fin.sum().item())
        rec = {"episodes": n_ep, "collect_success": (float((succ & fin).sum().item()) / n_ep) if n_ep else 0.0,
               "mean_reward": float(rewards[valid].mean().item()) if bool(valid.any()) else 0.0}
        idx = valid.reshape(-1).nonzero(as_tuple=False).squeeze(1)
        obs = obs_buf.reshape((-1,) + tuple(obs_buf.shape[2:]))[idx]
        return rec, obs, pi.reshape(-1, A)[idx], ret.reshape(-1)[idx], idx
