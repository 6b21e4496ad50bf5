"""On-device rollout collection — the data-collection half of twisterl's PPO loop (SURVEY.md §8f row 1).

The reference hands its envs to twisterl's PPO collector (rl/configs.py:133-137, 216-221: `num_episodes` cloned envs,
`reset()`, then `observe/masks -> policy -> sample -> step -> reward` until final, GAE(lambda, gamma) over each
episode, on a rayon pool of `num_cores`).  Here the B environments of one `BatchedEnv` play episodes back to back on
the GPU for `num_steps` decisions:

    reset_select (envs that are final start a new episode, Philox seed of this decision)
 -> observe (dense f32, device)  -> [twist: obs index i moves to obs_perms[k][i], k drawn per env]
 -> policy MLP (PyTorch) -> softmax -> [twist back: weights[g] = twisted_weights[act_perms[k][g]]]
 -> qg_collect_step: Philox inverse-CDF sample + fused env step + reward / done / success
 -> ... -> qg_gae over the [T][B] rollout.

Everything stays on the device; the result tensors are laid out [T, B, ...].  twisterl itself is not in the
reference tree, so its exact collector protocol is unpinned (SURVEY.md §8c); what is fixed here — and checked against
the CPU oracle in tests/test_collector.py — is the env side: which env resets when, which action each sample picks,
and the reward / done / advantage numbers that follow.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from ._lib import check, lib
from .engine import BatchedEnv, _dptr

SEED_STRIDE = 0x9E3779B97F4A7C15          # decision t of a collector seeded s uses Philox seed (s + t * SEED_STRIDE) mod 2^64


def decision_seed(seed: int, counter: int) -> int:
    return (seed + counter * SEED_STRIDE) & (2**64 - 1)


@dataclass
class Rollout:
    obs: torch.Tensor            # f32 [T, B, obs...]  what the policy saw (twisted when twists are on)
    actions: torch.Tensor        # i32 [T, B]          env action (-1: the env was final at decision time, slot unused)
    policy_actions: torch.Tensor  # i64 [T, B]         the same action in the policy's (twisted) action order
    logp: torch.Tensor           # f32 [T, B]          log pi(a | obs)
    values: torch.Tensor         # f32 [T+1, B]        V(obs_t); row T bootstraps truncated episodes
    rewards: torch.Tensor        # f32 [T, B]
    dones: torch.Tensor          # bool [T, B]         is_final after the step
    successes: torch.Tensor      # bool [T, B]
    valid: torch.Tensor          # bool [T, B]
    advantages: torch.Tensor     # f32 [T, B]
    returns: torch.Tensor        # f32 [T, B]
    twist: torch.Tensor | None   # i32 [T, B]          twist index used for the decision
    obs_bits: torch.Tensor | None = None   # i32 [T, B, obs_words]  packed observations (collect_packed: `obs` is None, unpack with unpack_obs)

    def unpack_obs(self, t0: int = 0, t1: int | None = None) -> torch.Tensor:
        """Dense f32 observations of decisions t0 .. t1-1 from the packed bits (for the update step of a trainer)."""
        return unpack_bits(self.obs_bits[t0:t1], self.obs_size)

    obs_size: int = 0

    def episode_stats(self):
        """(episodes finished, fraction of them that ended in success) over the rollout."""
        fin = self.dones & self.valid
        n = int(fin.sum().item())
        ok = int((self.successes & fin).sum().item())
        return n, (ok / n if n else 0.0)


def unpack_bits(bits: torch.Tensor, obs_size: int) -> torch.Tensor:
    """Packed observations int32 [..., obs_words] -> dense f32 [..., obs_size] (bit i % 32 of word i // 32 = entry i)."""
    shifts = torch.arange(32, dtype=torch.int32, device=bits.device)
    dense = ((bits.unsqueeze(-1) >> shifts) & 1).reshape(bits.shape[:-1] + (-1,))
    return dense[..., :obs_size].float()


def gae(rewards: torch.Tensor, values: torch.Tensor, dones: torch.Tensor, gamma: float, lam: float, valid: torch.Tensor | None = None):
    """qg_gae on [T, B] device tensors (values [T+1, B]); returns (advantages, returns)."""
    T, B = int(rewards.shape[0]), int(rewards.shape[1])
    assert rewards.is_cuda and rewards.dtype == torch.float32 and rewards.is_contiguous()
    assert values.shape == (T + 1, B) and values.dtype == torch.float32 and values.is_contiguous()
    assert dones.shape == (T, B) and dones.element_size() == 1 and dones.is_contiguous()
    assert valid is None or (valid.shape == (T, B) and valid.element_size() == 1 and valid.is_contiguous())
    adv = torch.empty_like(rewards)
    ret = torch.empty_like(rewards)
    st = C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)
    with torch.cuda.device(rewards.device):
        check(lib().qg_gae(_dptr(rewards), _dptr(values), _dptr(dones), _dptr(valid), T, B, C.c_float(gamma), C.c_float(lam), _dptr(adv), _dptr(ret), st))
    return adv, ret


def twist_gather(src: torch.Tensor, table: torch.Tensor, index: torch.Tensor | None, out: torch.Tensor | None = None):
    """out[b, j] = src[b, table[index[b], j]] (qg_twist_gather); src f32 [B, len] contiguous, table i32 [K, len]."""
    B = int(src.shape[0])
    flat = src.reshape(B, -1)
    assert flat.is_contiguous() and flat.dtype == torch.float32 and table.dtype == torch.int32 and table.is_contiguous()
    assert table.shape[1] == flat.shape[1]
    assert index is None or (index.dtype == torch.int32 and index.numel() == B)
    out = torch.empty_like(flat) if out is None else out
    st = C.c_void_p(torch.cuda.current_stream(src.device).cuda_stream)
    with torch.cuda.device(src.device):
        check(lib().qg_twist_gather(_dptr(flat), _dptr(out), _dptr(table), _dptr(index), B, int(flat.shape[1]), st))
    return out.reshape(src.shape)


def qubit_twist_table(obs_perms, num_qubits: int) -> np.ndarray:
    """uint8 [K, n]: the inverse qubit permutation of every twist, for qg_twist_bits.  Every obs perm of Permutation / LinearFunction /
    Clifford lifts a qubit permutation p to the d x d observation (d = n or 2n): entry (r, c) -> (lift(r), lift(c)), lift(i) = p[i] (i < n),
    n + p[i - n] (i >= n).  p is read off the first column and every row is checked to have that form."""
    op = np.asarray(obs_perms, dtype=np.int64)
    K, size = op.shape
    d, n = int(round(size ** 0.5)), int(num_qubits)
    if d * d != size or d not in (n, 2 * n):
        raise NotImplementedError(f"twists on packed observations need a square observation of side n or 2n (got {size} entries, n = {n})")
    p = op[:, : n * d : d] // d                                          # lift(i) for i < n, from entry (i, 0) -> (lift(i), lift(0))
    lift = p if d == n else np.concatenate([p, p + n], axis=1)
    if not np.array_equal(op, (lift[:, :, None] * d + lift[:, None, :]).reshape(K, size)) or not np.array_equal(np.sort(p, axis=1), np.broadcast_to(np.arange(n), p.shape)):
        raise NotImplementedError("an obs perm of these twists is not the lift of a qubit permutation: twists on packed observations do not apply")
    return np.argsort(p, axis=1).astype(np.uint8)


def twist_bits(src: torch.Tensor, out: torch.Tensor, qperm_inv: torch.Tensor, num_qubits: int, index: torch.Tensor | None = None,
               seed_dev: torch.Tensor | None = None, first_env_id: int = 0, draw: int = 0, index_out: torch.Tensor | None = None, obs_size: int | None = None):
    """qg_twist_bits: packed observations int32 [B, obs_words] -> the same observations in twist frame k[b] (entry i -> obs_perms[k][i]).
    k = index[b], or drawn on the device from the Philox seed in seed_dev (int64 [1]) — mulhi(philox(seed; first_env_id + b, draw, 5), K) —
    and written to index_out (int32 [B]) when given.  qperm_inv: uint8 [K, n] of qubit_twist_table."""
    B, ow = int(src.shape[0]), int(src.shape[-1])
    assert src.is_cuda and src.element_size() == 4 and src.is_contiguous() and out.is_contiguous() and out.shape == src.shape
    assert qperm_inv.dtype == torch.uint8 and qperm_inv.is_contiguous() and qperm_inv.shape[1] == num_qubits
    assert index is None or (index.dtype == torch.int32 and index.numel() == B)
    assert index is not None or (seed_dev is not None and seed_dev.element_size() == 8)
    assert index_out is None or (index_out.dtype == torch.int32 and index_out.numel() == B and index_out.is_contiguous())
    size = obs_size if obs_size is not None else ow * 32
    d = int(round(size ** 0.5))
    st = C.c_void_p(torch.cuda.current_stream(src.device).cuda_stream)
    with torch.cuda.device(src.device):
        check(lib().qg_twist_bits(_dptr(src), _dptr(out), B, int(size), int(num_qubits), d, _dptr(qperm_inv), int(qperm_inv.shape[0]), _dptr(index),
                                  _dptr(seed_dev), int(first_env_id), int(draw), _dptr(index_out), st))
    return out


class RolloutCollector:
    def __init__(self, env: BatchedEnv, policy: torch.nn.Module, gamma: float = 0.995, lam: float = 0.995, use_twists: bool = True,
                 seed: int = 0, first_env_id: int = 0, matmul_precision: str = "f32"):
        """matmul_precision: how PyTorch runs the policy's GEMMs while collecting — "f32" (the reference's arithmetic), "tf32" (tensor
        cores, f32 accumulate; the observations are 0/1 and exact, only the weights are rounded to 10 mantissa bits) or "bf16"
        (autocast).  The env side is unaffected; only the action probabilities the samples are drawn from change in their last bits."""
        assert matmul_precision in ("f32", "tf32", "bf16")
        self.matmul_precision = matmul_precision
        self.env, self.policy = env, policy.to(env.device).eval()
        self.gamma, self.lam = float(gamma), float(lam)
        self.seed, self.first_env_id = int(seed), int(first_env_id)
        self.counter = 0                  # decisions made so far: decision t draws from decision_seed(seed, t)
        self.obs_table = self.act_table = None
        if use_twists:
            obs_perms, act_perms = env.twists()
            if len(obs_perms) > 1:
                op = np.asarray(obs_perms, dtype=np.int64)
                inv = np.empty_like(op)
                rows = np.arange(op.shape[0])[:, None]
                inv[rows, op] = np.arange(op.shape[1])[None, :]          # entry i moves to obs_perms[k][i]  <=>  out[j] = in[inv[k][j]]
                self.obs_table = torch.from_numpy(inv.astype(np.int32)).to(env.device)
                self.act_table = torch.from_numpy(np.asarray(act_perms, dtype=np.int32)).to(env.device)
        self.num_twists = 0 if self.obs_table is None else int(self.obs_table.shape[0])
        self.qperm_table = None           # collect_packed: uint8 [K, n] inverse qubit permutations (qubit_twist_table), built on first use
        self._gen = torch.Generator(device=env.device)
        self._gen.manual_seed(self.seed & (2**63 - 1))
        self.hook = None                  # tests: called as hook(t, weights [B, A] in env action order) before each collect step
        self._packed = {}                 # collect_packed: buffers / CUDA graph per (num_steps, deterministic)

    def _policy(self, obs):
        with torch.no_grad():
            if self.matmul_precision == "bf16":
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    logits, value = self.policy(obs)
            elif self.matmul_precision == "tf32":
                prev = torch.backends.cuda.matmul.allow_tf32
                torch.backends.cuda.matmul.allow_tf32 = True
                try:
                    logits, value = self.policy(obs)
                finally:
                    torch.backends.cuda.matmul.allow_tf32 = prev
            else:
                logits, value = self.policy(obs)
            return torch.softmax(logits.float(), dim=-1), value.float().reshape(-1)

    def tensor_core_policy(self):
        """The collect_packed policy handle (policy.TensorCorePolicy) refreshed from self.policy (TensorCorePolicy.refresh): a weight update
        (optimizer step, load_state_dict) is copied into the handle in place, so captured rollout graphs stay valid; they are dropped when the
        handle is recreated (another module that cannot be loaded in place) or rebuilt for a larger batch.
        Raises NotImplementedError where the tensor-core policy cannot run (more than 127 actions, a value head that is not one Linear,
        a device that is not sm_100)."""
        from .policy import TensorCorePolicy
        B = self.env.batch
        tcp = getattr(self, "_tcp", None)
        if tcp is None or tcp.max_batch < B:
            tcp = self._tcp = TensorCorePolicy(self.policy, max_batch=B, device=self.env.device, with_value=True)
            self._packed = {}
        elif tcp.refresh(self.policy):
            self._packed = {}
        return tcp

    def collect_packed(self, num_steps: int, deterministic: bool = False, use_cuda_graph: bool = True) -> Rollout:
        """The large-batch collection path: packed-bit observations (32x less observation traffic than dense f32) and the policy on the
        tensor cores (policy.TensorCorePolicy, tcgen05).  Per decision: reset_select -> observe_bits [-> qg_twist_bits: the observation in a
        twist frame drawn per env on the device] -> qg_policy_tc_forward_bits (softmax weights + value) -> qg_collect_step (twisted collectors:
        qg_collect_step_twisted_dev, which maps the policy's actions back to the env's order while it samples); log-probabilities and GAE once
        at the end.  Same contract as collect(): obs_bits hold what the policy saw, `twist` the twist indices, policy_actions the action in the
        policy's order.  Twist k of env b at decision t is mulhi(philox(decision seed t; first_env_id + b, 0, stream 5), K); the bootstrap
        observation after the last decision uses draw 1 of the last decision's seed.
        use_cuda_graph: the whole rollout (num_steps decisions, ~6 launches each) is captured once and replayed; the decisions' Philox seeds
        are read from a device array the host refills before every replay (qg_reset_select_dev / qg_collect_step_dev).  A weight update is
        loaded into the policy handle in place, so the graph survives training steps.  The returned tensors are the collector's own buffers:
        they are overwritten by the next call with the same num_steps."""
        env, T, B = self.env, int(num_steps), self.env.batch
        dev, A = env.device, env.num_actions()
        assert T >= 1
        twisted = self.num_twists > 0
        if twisted and self.qperm_table is None:
            self.qperm_table = torch.from_numpy(qubit_twist_table(env.twists()[0], int(env.cfg.num_qubits))).to(dev)
        tcp = self.tensor_core_policy()
        st = self._packed.get((T, deterministic))
        if st is None:
            ow = env.obs_words()
            st = {"bits": torch.empty((T + 1, B, ow), dtype=torch.int32, device=dev), "probs": torch.empty((T, B, A), dtype=torch.float32, device=dev),
                  "actions": torch.full((T, B), -1, dtype=torch.int32, device=dev), "rewards": torch.zeros((T, B), dtype=torch.float32, device=dev),
                  "dones": torch.zeros((T, B), dtype=torch.bool, device=dev), "succ": torch.zeros((T, B), dtype=torch.bool, device=dev),
                  "values": torch.zeros((T + 1, B), dtype=torch.float32, device=dev), "seeds": torch.zeros(T, dtype=torch.int64, device=dev),
                  "seeds_host": torch.zeros(T, dtype=torch.int64).pin_memory(), "graph": None, "runs": 0}
            if twisted:
                st["raw"] = torch.empty((B, ow), dtype=torch.int32, device=dev)                  # observe_bits before the twist
                st["twist"] = torch.zeros((T + 1, B), dtype=torch.int32, device=dev)            # row T: the bootstrap observation's twist
                st["pol_actions"] = torch.full((T, B), -1, dtype=torch.int32, device=dev)
            self._packed[(T, deterministic)] = st
        difficulty = env.difficulty
        if st.get("difficulty") != difficulty:       # the env config (difficulty included) is a launch parameter a captured graph keeps
            st["graph"], st["runs"], st["difficulty"] = None, 0, difficulty
        bits, probs, actions, rewards, dones, succ, values, seeds = (st[k] for k in ("bits", "probs", "actions", "rewards", "dones", "succ", "values", "seeds"))
        for t in range(T):          # the seeds of this rollout's decisions (two's-complement view of the uint64 seeds)
            s_ = decision_seed(self.seed, self.counter + t)
            st["seeds_host"][t] = s_ - (1 << 64) if s_ >= (1 << 63) else s_
        seeds.copy_(st["seeds_host"], non_blocking=True)
        self.counter += T
        n = int(env.cfg.num_qubits)

        def observe(t, draw, seed_row):
            if not twisted:
                env.observe_bits(bits[t])
                return
            env.observe_bits(st["raw"])
            twist_bits(st["raw"], bits[t], self.qperm_table, n, seed_dev=seeds[seed_row:seed_row + 1], first_env_id=self.first_env_id, draw=draw,
                       index_out=st["twist"][t], obs_size=env._obs_size)

        def body():
            for t in range(T):
                env.reset_select_dev(seeds[t:t + 1], self.first_env_id)
                observe(t, 0, t)
                tcp.forward_bits(bits[t], probs=probs[t], values=values[t])
                if twisted:
                    env.collect_step_twisted_dev(probs[t], self.act_table, st["twist"][t], seeds[t:t + 1], deterministic=deterministic, chosen=actions[t],
                                                 policy_chosen=st["pol_actions"][t], reward=rewards[t], done=dones[t], success=succ[t])
                else:
                    env.collect_step_dev(probs[t], seeds[t:t + 1], deterministic=deterministic, chosen=actions[t], reward=rewards[t], done=dones[t], success=succ[t])
            observe(T, 1, T - 1)
            tcp.forward_bits(bits[T], values=values[T])

        if not use_cuda_graph:
            body()
        elif st["graph"] is None and st["runs"] == 0:
            body()                                  # the first rollout runs eagerly (lazy initialisation outside any capture) ...
            st["runs"] = 1
        else:
            if st["graph"] is None:                 # ... the second one is captured, then replayed
                torch.cuda.current_stream(dev).synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    body()
                st["graph"] = g
            st["graph"].replay()
        valid = actions >= 0
        a = (st["pol_actions"] if twisted else actions).long().clamp_(min=0)
        logp = torch.log(probs.gather(2, a[..., None]).squeeze(2).clamp_min(1e-38))
        adv, ret = gae(rewards, values, dones, self.gamma, self.lam, valid)
        return Rollout(obs=None, actions=actions, policy_actions=a, logp=logp, values=values, rewards=rewards, dones=dones, successes=succ, valid=valid,
                       advantages=adv, returns=ret, twist=st["twist"][:T] if twisted else None, obs_bits=bits[:T], obs_size=env._obs_size)

    def collect(self, num_steps: int, deterministic: bool = False) -> Rollout:
        env, T, B = self.env, int(num_steps), self.env.batch
        dev = env.device
        obs_buf = torch.empty((T, B) + tuple(env.obs_shape()), dtype=torch.float32, device=dev)
        actions = torch.full((T, B), -1, dtype=torch.int32, device=dev)
        rewards = torch.zeros((T, B), dtype=torch.float32, device=dev)
        dones = torch.zeros((T, B), dtype=torch.bool, device=dev)
        succ = torch.zeros((T, B), dtype=torch.bool, device=dev)
        values = torch.zeros((T + 1, B), dtype=torch.float32, device=dev)
        logp = torch.zeros((T, B), dtype=torch.float32, device=dev)
        pol_actions = torch.zeros((T, B), dtype=torch.int64, device=dev)
        twist = torch.zeros((T, B), dtype=torch.int32, device=dev) if self.num_twists else None
        raw = torch.empty((B,) + tuple(env.obs_shape()), dtype=torch.float32, device=dev) if self.num_twists else None
        direct = (B * env._obs_size * 4) % 16 == 0        # the engine wants 16-byte aligned observation tensors
        for t in range(T):
            s = decision_seed(self.seed, self.counter)
            # episodes that ended (or a fresh collector: every env, the constructor state is final) start over
            env.reset_select(s, self.first_env_id)
            kidx = None
            if self.num_twists:
                kidx = torch.randint(0, self.num_twists, (B,), generator=self._gen, device=dev, dtype=torch.int32)
                twist[t] = kidx
                env.observe(out=raw)
                twist_gather(raw, self.obs_table, kidx, out=obs_buf[t].reshape(B, -1))
            elif direct:
                env.observe(out=obs_buf[t])
            else:
                obs_buf[t].copy_(env.observe())
            probs_tw, values[t] = self._policy(obs_buf[t])
            probs = probs_tw if kidx is None else twist_gather(probs_tw.contiguous(), self.act_table, kidx)
            probs = probs.contiguous()
            if self.hook is not None:
                self.hook(t, probs)
            env.collect_step(probs, s, deterministic=deterministic, obs=False, chosen=actions[t], reward=rewards[t], done=dones[t], success=succ[t])
            a = actions[t].long().clamp_(min=0)
            logp[t] = torch.log(probs.gather(1, a[:, None]).squeeze(1).clamp_min(1e-38))
            pol_actions[t] = a if kidx is None else self.act_table[kidx.long(), a].long()
            self.counter += 1
        # bootstrap value for the episodes cut by the end of the rollout (V of the observation after the last step)
        kidx = None
        if self.num_twists:
            kidx = torch.randint(0, self.num_twists, (B,), generator=self._gen, device=dev, dtype=torch.int32)
            env.observe(out=raw)
            last = twist_gather(raw, self.obs_table, kidx)
        else:
            last = env.observe()
        _, values[T] = self._policy(last)
        valid = actions >= 0
        adv, ret = gae(rewards, values, dones, self.gamma, self.lam, valid)
        return Rollout(obs=obs_buf, actions=actions, policy_actions=pol_actions, logp=logp, values=values, rewards=rewards, dones=dones,
                       successes=succ, valid=valid, advantages=adv, returns=ret, twist=twist)
