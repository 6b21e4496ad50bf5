"""The packed tensor-core collector with twists (RolloutCollector.collect_packed): twisted packed observations (qg_twist_bits), the twisted
collect step (qg_collect_step_twisted_dev), in-place weight refresh of the tensor-core policy (qg_policy_tc_load_weights_dev) and PPO
on that path (matmul_precision="tensor_core").  The env side is re-enacted with the CPU oracle, as in tests/test_collector.py."""
import copy

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_collector import cpu_gae, dense
from tests.test_search import STREAM_SAMPLE, cpu_pick

STREAM_TWIST = 5


def configs():
    t = H.config_table()
    out = {name: t[name] for name in ("C1_perm_grid3", "clifford3_allgates", "lf5_line_swap")}
    n, gs = H.gateset_from_coupling_map([(i, j) for i in range(5) for j in range(5) if i != j], ("H", "S", "CX"))
    out["clifford5_all_to_all"] = (H.CLIFF, n, gs, {})
    return out


TWIST_CONFIGS = ["C1_perm_grid3", "clifford3_allgates", "lf5_line_swap", "clifford5_all_to_all"]


def inverse_obs_table(obs_perms):
    op = np.asarray(obs_perms, dtype=np.int64)
    inv = np.empty_like(op)
    inv[np.arange(op.shape[0])[:, None], op] = np.arange(op.shape[1])[None, :]
    return inv.astype(np.int32)


def mulhi(raw, K):
    return (int(raw) * int(K)) >> 32


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", TWIST_CONFIGS)
def test_qubit_twist_table_lifts_to_obs_perms(name):
    """The [K][n] table of inverse qubit permutations, lifted back to the d x d observation, is exactly the inverse of every obs perm."""
    from qiskit_gym_b200.collector import qubit_twist_table
    kind, n, gs, kw = configs()[name]
    env = orc.OracleEnv(kind, n, gs, **dict(kw, add_inverts=False, add_perms=True))
    obs_perms, _ = env.twists()
    qpinv = qubit_twist_table(obs_perms, n).astype(np.int64)
    K, size = np.asarray(obs_perms).shape
    if name == "clifford5_all_to_all":
        assert K == 120
    d = int(round(size ** 0.5))
    liftinv = qpinv if d == n else np.concatenate([qpinv, qpinv + n], axis=1)
    table = (liftinv[:, :, None] * d + liftinv[:, None, :]).reshape(K, size)
    assert np.array_equal(table, inverse_obs_table(obs_perms))


def test_qubit_twist_table_rejects_other_perms():
    from qiskit_gym_b200.collector import qubit_twist_table
    op = np.tile(np.arange(9), (2, 1))
    op[1, [0, 1]] = [1, 0]                      # swaps two entries of one row: no qubit permutation does that
    with pytest.raises(NotImplementedError):
        qubit_twist_table(op.tolist(), 3)


# ---------------------------------------------------------------------------------------------------- GPU
def make_env(name, B, **extra):
    from qiskit_gym_b200 import BatchedEnv
    kind, n, gs, kw = configs()[name]
    ekw = dict(kw, add_inverts=False, add_perms=True, **extra)
    return BatchedEnv(kind, n, gs, B, **ekw), (kind, n, gs, ekw)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TWIST_CONFIGS)
def test_twist_bits_matches_dense_gather(name):
    from qiskit_gym_b200.collector import qubit_twist_table, twist_bits, twist_gather
    from qiskit_gym_b200.policy import pack_obs_bits
    B, first, seed = 1000, 321, 0xDEADBEEF12345
    env, (kind, n, gs, _) = make_env(name, B, difficulty=4)
    dev = env.device
    env.reset(seed=7, first_env_id=first)
    obs_perms, _ = env.twists()
    K = len(obs_perms)
    qpinv = torch.from_numpy(qubit_twist_table(obs_perms, n)).to(dev)
    inv = torch.from_numpy(inverse_obs_table(obs_perms)).to(dev)
    raw = env.observe_bits(env.new_obs_bits())
    dense_obs = env.observe().reshape(B, -1).contiguous()
    size = dense_obs.shape[1]
    rng = np.random.Generator(np.random.PCG64(4))
    # given indices
    k = torch.from_numpy(rng.integers(K, size=B).astype(np.int32)).to(dev)
    out = torch.full_like(raw, -1)
    twist_bits(raw, out, qpinv, n, index=k, obs_size=size)
    want = pack_obs_bits(twist_gather(dense_obs, inv, k))
    assert torch.equal(out.cpu(), want)
    # drawn indices: mulhi(philox(seed; first + b, draw, 5), K), and the bits in those frames
    seed_dev = torch.tensor([seed], dtype=torch.int64, device=dev)
    for draw in (0, 1):
        kout = torch.full((B,), -1, dtype=torch.int32, device=dev)
        twist_bits(raw, out, qpinv, n, seed_dev=seed_dev, first_env_id=first, draw=draw, index_out=kout, obs_size=size)
        kk = kout.cpu().numpy()
        assert [int(x) for x in kk] == [mulhi(orc.philox_draw(seed, first + b, draw, STREAM_TWIST), K) for b in range(B)]
        assert torch.equal(out.cpu(), pack_obs_bits(twist_gather(dense_obs, inv, kout)))
        if K > 1:
            assert len(set(kk.tolist())) > 1
        # two halves with first_env_id offsets draw what one batch draws
        h = B // 2
        parts = []
        for lo, hi in ((0, h), (h, B)):
            kp = torch.full((hi - lo,), -1, dtype=torch.int32, device=dev)
            op = torch.empty_like(raw[lo:hi])
            twist_bits(raw[lo:hi].contiguous(), op, qpinv, n, seed_dev=seed_dev, first_env_id=first + lo, draw=draw, index_out=kp, obs_size=size)
            parts.append(kp)
        assert torch.equal(torch.cat(parts), kout)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TWIST_CONFIGS)
@pytest.mark.parametrize("deterministic", [False, True])
def test_twisted_collect_step_matches_gather(name, deterministic):
    """qg_collect_step_twisted_dev == qg_twist_gather(weights, act_perms, k) + qg_collect_step_dev, bit for bit."""
    from qiskit_gym_b200.collector import decision_seed, twist_gather
    B, first = 1024, 40
    envs = [make_env(name, B, difficulty=5, max_depth=8, depth_slope=2)[0] for _ in range(2)]
    dev = envs[0].device
    A = envs[0].num_actions()
    _, act_perms = envs[0].twists()
    act = torch.tensor(act_perms, dtype=torch.int32, device=dev)
    K = act.shape[0]
    rng = np.random.Generator(np.random.PCG64(8))
    for e in envs:
        e.reset(seed=99, first_env_id=first)
    stepped = 0
    for t in range(6):
        s = decision_seed(5, t)
        seed_dev = torch.tensor([s - (1 << 64) if s >= (1 << 63) else s], dtype=torch.int64, device=dev)
        for e in envs:
            e.reset_select_dev(seed_dev, first)
        w = torch.from_numpy(rng.random((B, A)).astype(np.float32) ** 3).to(dev)
        w /= w.sum(1, keepdim=True)
        k = torch.from_numpy(rng.integers(K, size=B).astype(np.int32)).to(dev)
        outs = [[torch.full((B,), -1, dtype=torch.int32, device=dev), torch.zeros(B, device=dev), torch.zeros(B, dtype=torch.bool, device=dev),
                 torch.zeros(B, dtype=torch.bool, device=dev)] for _ in envs]
        pol = torch.full((B,), -7, dtype=torch.int32, device=dev)
        envs[0].collect_step_twisted_dev(w, act, k, seed_dev, deterministic=deterministic, chosen=outs[0][0], policy_chosen=pol,
                                         reward=outs[0][1], done=outs[0][2], success=outs[0][3])
        envs[1].collect_step_dev(twist_gather(w, act, k).contiguous(), seed_dev, deterministic=deterministic, chosen=outs[1][0], reward=outs[1][1],
                                 done=outs[1][2], success=outs[1][3])
        assert torch.equal(outs[0][0], outs[1][0])
        assert torch.equal(outs[0][1].view(torch.int32), outs[1][1].view(torch.int32))
        assert torch.equal(outs[0][2], outs[1][2]) and torch.equal(outs[0][3], outs[1][3])
        ch = outs[0][0].long()
        on = ch >= 0
        stepped += int(on.sum())
        assert torch.equal(pol[~on], torch.full_like(pol[~on], -1))
        assert torch.equal(pol[on], act[k.long()[on], ch[on]])
        for b in (0, 1, 17, 500, B - 1):
            assert np.array_equal(envs[0].get_state(b), envs[1].get_state(b))
    assert stepped > B


def reenact(ro, spec, tcp, act_perms, obs_perms, seed, first, T, B, gamma, lam, rows=None):
    """The rollout re-enacted with the oracle: resets, (twisted) observations, samples from the recomputed tensor-core probabilities, rewards, GAE.
    rows: re-enact only these envs (envs are independent by (seed, env id)); all B by default."""
    from qiskit_gym_b200.collector import decision_seed
    kind, n, gs, ekw = spec
    rows = list(range(B)) if rows is None else [int(b) for b in rows]
    refs = [orc.OracleEnv(kind, n, gs, **ekw) for _ in rows]
    ticks = np.zeros(len(rows), np.int64)
    acts, pacts = ro.actions.cpu().numpy()[:, rows], ro.policy_actions.cpu().numpy()[:, rows]
    rew, dones, succ = ro.rewards.cpu().numpy()[:, rows], ro.dones.cpu().numpy()[:, rows], ro.successes.cpu().numpy()[:, rows]
    obs = ro.unpack_obs().cpu().numpy()[:, rows]
    size = obs.shape[-1]
    tw = None if ro.twist is None else ro.twist.cpu().numpy()[:, rows]
    K = len(obs_perms) if obs_perms is not None else 1
    n_resets = 0
    for t in range(T):
        s = decision_seed(seed, t)
        probs = tcp.forward_bits(ro.obs_bits[t].contiguous()).cpu().numpy()[rows]
        for i, (b, r) in enumerate(zip(rows, refs)):
            if r.is_final():
                r.reset(seed=s, env_id=first + b)
                ticks[i] = 0
                n_resets += 1
            want = dense(r.observe(), size)
            if tw is not None:
                k = int(tw[t, i])
                assert k == mulhi(orc.philox_draw(s, first + b, 0, STREAM_TWIST), K)
                tmp = np.zeros(size, np.float32)
                tmp[np.asarray(obs_perms[k])] = want
                want = tmp
            assert np.array_equal(obs[t, i], want), (t, b)
            if r.is_final():
                assert acts[t, i] == -1
                continue
            w = probs[i] if tw is None else probs[i][np.asarray(act_perms[int(tw[t, i])])]
            a = cpu_pick(w, orc.philox_draw(s, first + b, int(ticks[i]), STREAM_SAMPLE), False)
            assert acts[t, i] == a, (t, b)
            assert pacts[t, i] == (a if tw is None else act_perms[int(tw[t, i])][a])
            r.step(a)
            ticks[i] += 1
            assert np.float32(r.reward()).view(np.uint32) == rew[t, i].view(np.uint32)
            assert bool(dones[t, i]) == r.is_final() and bool(succ[t, i]) == r.success()
    assert n_resets > len(rows) if len(rows) == B else n_resets >= len(rows)
    valid = acts >= 0
    assert np.array_equal(ro.valid.cpu().numpy()[:, rows], valid)
    ra, rr = cpu_gae(rew, ro.values.cpu().numpy()[:, rows], dones, valid, gamma, lam)
    assert np.array_equal(ro.advantages.cpu().numpy()[:, rows].view(np.uint32), ra.view(np.uint32))
    assert np.array_equal(ro.returns.cpu().numpy()[:, rows].view(np.uint32), rr.view(np.uint32))
    lp = np.log(np.take_along_axis(np.stack([tcp.forward_bits(ro.obs_bits[t].contiguous()).cpu().numpy()[rows] for t in range(T)]),
                                   np.maximum(pacts, 0)[..., None].astype(np.int64), axis=2)[..., 0])
    assert np.allclose(ro.logp.cpu().numpy()[:, rows][valid], lp[valid], rtol=1e-5, atol=1e-6)


def rollout_fields(ro):
    out = [ro.actions, ro.policy_actions, ro.rewards.view(torch.int32), ro.dones, ro.successes, ro.values.view(torch.int32), ro.obs_bits,
           ro.advantages.view(torch.int32), ro.logp.view(torch.int32)]
    return [x.clone() for x in out] + ([ro.twist.clone()] if ro.twist is not None else [])


@pytest.mark.gpu
@pytest.mark.parametrize("name,twists", [("C1_perm_grid3", True), ("clifford3_allgates", True), ("lf5_line_swap", True), ("lf5_line_swap", False),
                                         ("clifford5_all_to_all", True)])
def test_collect_packed_matches_cpu_reenactment(name, twists):
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.search import BasicPolicy

    kind, n, gs, kw = configs()[name]
    ekw = dict(kw, add_inverts=False, add_perms=twists, difficulty=2, max_depth=5, depth_slope=2)
    B, T, seed, first, gamma, lam = 70, 24, 1234, 500, 0.99, 0.9
    env = BatchedEnv(kind, n, gs, B, **ekw)
    torch.manual_seed(0)
    pol = BasicPolicy(env.obs_shape(), len(gs), embedding_size=64, common_layers=(32,))
    col = RolloutCollector(env, pol, gamma=gamma, lam=lam, use_twists=twists, seed=seed, first_env_id=first)
    assert (col.num_twists > 1) == twists
    ro = col.collect_packed(T, use_cuda_graph=False)
    assert (ro.twist is not None) == twists
    obs_perms, act_perms = env.twists() if twists else (None, None)
    reenact(ro, (kind, n, gs, ekw), col._tcp, act_perms, obs_perms, seed, first, T, B, gamma, lam)
    if twists:                 # the bootstrap observation's twist (row T of the collector's buffer)
        from qiskit_gym_b200.collector import decision_seed
        st = col._packed[(T, False)]
        K = len(obs_perms)
        s = decision_seed(seed, T - 1)
        assert [int(x) for x in st["twist"][T].cpu()] == [mulhi(orc.philox_draw(s, first + b, 1, STREAM_TWIST), K) for b in range(B)]


@pytest.mark.gpu
@pytest.mark.parametrize("twists", [True, False])
def test_collect_packed_graph_replay_equals_eager(twists):
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.search import BasicPolicy
    B, T = 2000, 6
    envs = [make_env("clifford3_allgates", B, difficulty=3, max_depth=6, depth_slope=2)[0] for _ in range(2)]
    torch.manual_seed(1)
    pol = BasicPolicy(envs[0].obs_shape(), envs[0].num_actions(), embedding_size=128, common_layers=(64,))
    cols = [RolloutCollector(e, pol, use_twists=twists, seed=77, first_env_id=9) for e in envs]
    for it in range(3):
        got = [rollout_fields(cols[0].collect_packed(T, use_cuda_graph=False)), rollout_fields(cols[1].collect_packed(T, use_cuda_graph=True))]
        for a, b in zip(*got):
            assert torch.equal(a, b), it
    assert cols[1]._packed[(T, False)]["graph"] is not None


def _adam_step(pol, seed):
    torch.manual_seed(seed)
    opt = torch.optim.Adam(pol.parameters(), lr=1e-2)
    dev = next(pol.parameters()).device
    x = (torch.rand((64, pol.embeddings.in_features), device=dev) < 0.3).float()
    logits, v = pol(x)
    loss = logits.square().mean() + v.square().mean()
    opt.zero_grad()
    loss.backward()
    opt.step()


@pytest.mark.gpu
@pytest.mark.parametrize("per_layer", [False, True])
def test_load_weights_equals_fresh_handle(per_layer):
    from qiskit_gym_b200.policy import TensorCorePolicy, pack_obs_bits
    from qiskit_gym_b200.search import BasicPolicy
    dev = torch.device("cuda", 0)
    torch.manual_seed(2)
    pol = BasicPolicy([16, 16], 72, embedding_size=512, common_layers=(256,)).to(dev)
    B = 3000
    tcp = TensorCorePolicy(pol, max_batch=B, device=dev)
    assert tcp.set_per_layer(per_layer) == (not per_layer)           # this network fits the fused kernel
    bits = pack_obs_bits(torch.from_numpy((np.random.Generator(np.random.PCG64(1)).random((B, 256)) < 0.5).astype(np.float32))).to(dev)

    def run(h):
        p, lg, v = torch.empty((B, 72), device=dev), torch.empty((B, 72), device=dev), torch.empty(B, device=dev)
        h.forward_bits(bits, probs=p, logits=lg, values=v)
        return [x.view(torch.int32).clone() for x in (p, lg, v)]

    before = run(tcp)
    _adam_step(pol, 3)
    tcp.load_weights(pol)
    fresh = TensorCorePolicy(pol, max_batch=B, device=dev)
    fresh.set_per_layer(per_layer)
    after, want = run(tcp), run(fresh)
    assert not torch.equal(before[0], after[0])
    for a, b in zip(after, want):
        assert torch.equal(a, b)
    # shapes that differ from creation are rejected
    other = BasicPolicy([16, 16], 72, embedding_size=256, common_layers=(256,)).to(dev)
    assert not tcp.can_load(other)
    with pytest.raises(ValueError):
        tcp.load_weights(other)


@pytest.mark.gpu
@pytest.mark.parametrize("twists", [True, False])
def test_graph_captured_before_update_replays_new_weights(twists):
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.search import BasicPolicy
    B, T = 1500, 5
    envs = [make_env("C1_perm_grid3", B, difficulty=3, max_depth=6, depth_slope=2)[0] for _ in range(2)]
    torch.manual_seed(4)
    pol = BasicPolicy(envs[0].obs_shape(), envs[0].num_actions(), embedding_size=128, common_layers=(64,)).to(envs[0].device)
    cg = RolloutCollector(envs[0], pol, use_twists=twists, seed=5, first_env_id=0)
    ce = RolloutCollector(envs[1], pol, use_twists=twists, seed=5, first_env_id=0)
    for _ in range(2):
        cg.collect_packed(T, use_cuda_graph=True)
        ce.collect_packed(T, use_cuda_graph=False)
    graph, tcp = cg._packed[(T, False)]["graph"], cg._tcp
    assert graph is not None
    _adam_step(pol, 6)
    a = rollout_fields(cg.collect_packed(T, use_cuda_graph=True))
    b = rollout_fields(ce.collect_packed(T, use_cuda_graph=False))
    assert cg._packed[(T, False)]["graph"] is graph and cg._tcp is tcp          # refreshed in place: same handle, same graph
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_ppo_tensor_core_learns_permutation_line4(tmp_path):
    """test_ppo.py::test_ppo_learns_permutation_line4 on the packed tensor-core collector, twists on."""
    from qiskit_gym_b200.specs import SynthSpec
    from qiskit_gym_b200.rl import RLSynthesis

    torch.manual_seed(0)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], difficulty=1, depth_slope=2, max_depth=32)
    cfg = {"collecting": {"num_episodes": 512}, "training": {"num_epochs": 4, "ent_coef": 0.01}, "optimizer": {"lr": 2e-3},
           "learning": {"diff_threshold": 0.85, "diff_max": 8, "diff_metric": "ppo_deterministic"},
           "evals": {"ppo_deterministic": {"num_episodes": 128}}, "logging": {"log_freq": 1, "checkpoint_freq": 20}}
    rls = RLSynthesis(env, cfg, {"embedding_size": 64, "common_layers": [64]}, device=0)
    targets = [list(np.random.Generator(np.random.PCG64(s)).permutation(4)) for s in range(24)]
    targets = [t for t in targets if t != [0, 1, 2, 3]]
    before = sum(rls.synth(t, deterministic=True, num_searches=1) is not None for t in targets)
    hist = rls.learn(initial_difficulty=1, num_iterations=40, tb_path=str(tmp_path), matmul_precision="tensor_core")
    assert len(hist) == 40 and hist[-1]["difficulty"] >= 4, [(h["difficulty"], round(h["eval/ppo_deterministic"], 2)) for h in hist]
    after = sum(rls.synth(t, deterministic=True, num_searches=1) is not None for t in targets)
    assert after >= max(before + 5, int(0.8 * len(targets))), (before, after, len(targets))


@pytest.mark.gpu
def test_ppo_update_on_packed_bits_equals_dense():
    from qiskit_gym_b200.collector import Rollout
    from qiskit_gym_b200.ppo import PPO
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = configs()["C1_perm_grid3"]
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=128, common_layers=(64,))
    cfg = {"collecting": {"num_episodes": 600}, "training": {"num_epochs": 3}}
    ppo = PPO(kind, n, gs, pol, cfg, device=0, seed=3, matmul_precision="tensor_core", difficulty=3, **dict(kw, add_perms=True))
    ro = ppo.collector.collect_packed(ppo._episode_steps())
    assert ro.obs is None and ro.twist is not None
    dense_ro = Rollout(obs=ro.unpack_obs().reshape(ro.actions.shape + (n, n)), actions=ro.actions, policy_actions=ro.policy_actions, logp=ro.logp,
                       values=ro.values, rewards=ro.rewards, dones=ro.dones, successes=ro.successes, valid=ro.valid, advantages=ro.advantages,
                       returns=ro.returns, twist=ro.twist)
    p0, o0 = copy.deepcopy(ppo.policy.state_dict()), copy.deepcopy(ppo.opt.state_dict())
    s_packed = ppo.update(ro)
    ppo.policy.load_state_dict(p0)
    ppo.opt.load_state_dict(o0)
    s_dense = ppo.update(dense_ro)
    assert s_packed == s_dense


@pytest.mark.gpu
def test_ppo_tensor_core_rejects_unsupported():
    from qiskit_gym_b200.ppo import PPO
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = configs()["C1_perm_grid3"]
    cfg = {"collecting": {"num_episodes": 64}}
    with pytest.raises(NotImplementedError):          # value head that is not one Linear
        PPO(kind, n, gs, BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,), value_layers=(16,)), cfg, device=0,
            matmul_precision="tensor_core", **kw)
    m = 17                                            # 136 SWAP actions: more than the tensor-core head's 127
    _, big = H.gateset_from_coupling_map([(i, j) for i in range(m) for j in range(i + 1, m)], ("SWAP",))
    with pytest.raises(NotImplementedError):
        PPO(H.PERM, m, big, BasicPolicy([m, m], len(big), embedding_size=64, common_layers=(32,)), cfg, device=0, use_twists=False,
            matmul_precision="tensor_core")
    with pytest.raises(ValueError):
        PPO(kind, n, gs, BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,)), cfg, device=0, matmul_precision="fp8", **kw)
