"""The twisted tree search (MCTSSearch(use_twists=True), csrc/qg_mcts.cu) and AlphaZero self-play on it (AlphaZero(use_twists=True)).

Protocol, restated: tree i belongs to the rollout with global id g = first + i; evaluation e = 0 is its root, e = s + 1 the leaf created by
simulation s.  The evaluation runs in frame  k(i, e) = mulhi(philox(seed; g + (e << 32), tick_i, 5), K)  (tick_i: the rollout's step counter
at decision time, K: the env's twists with add_perms); the policy sees the node's observation moved by obs_perms[k], and the node stores
P(a) = probs[act_perm[k][a]].  The value is used as is; PUCT, back-up, root weights, re-rooting and the decision are those of the
untwisted search.  The policy outputs are recorded on the GPU and the trees re-enacted on the CPU with the oracle's envs and twists."""
import inspect

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_mcts import CpuTree
from tests.test_mcts_reuse import NODE_FIELDS, ReuseTree, env_key, reroot
from tests.test_search import STREAM_SAMPLE, cpu_pick
from tests.test_search_many import _replays_to_success

STREAM_TWIST = 5
f32 = np.float32


def frame(seed, g, e, tick, K):
    return (orc.philox_draw(seed, g + (e << 32), tick, STREAM_TWIST) * K) >> 32


def _pack(indices, obs):
    bits = np.zeros((obs + 31) // 32 * 32, dtype=np.uint8)
    bits[list(indices)] = 1
    return np.packbits(bits, bitorder="little").view(np.uint32)


# ---- CPU: refusals before any allocation -------------------------------------------------------------------------------------------
def _no_device(monkeypatch):
    import qiskit_gym_b200.mcts as mcts
    import qiskit_gym_b200.ppo as ppo

    def refuse(*a, **k):
        raise AssertionError("an engine was allocated before the refusal")
    monkeypatch.setattr(mcts, "BatchedEnv", refuse)
    monkeypatch.setattr(ppo, "BatchedEnv", refuse)


def test_refusals_before_any_device_work(monkeypatch):
    """MCTSSearch(use_twists=True) and AlphaZero(use_twists=True) refuse the torch backend, a policy without single-Linear heads,
    PauliNetwork and a Permutation wider than 64 qubits (NotImplementedError), and add_perms=False (ValueError), before any engine."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.ppo import AlphaZero
    from qiskit_gym_b200.search import BasicPolicy
    _no_device(monkeypatch)
    kind, n, gs, _ = H.config_table()["C1_perm_grid3"]
    pol = BasicPolicy([n, n], len(gs), embedding_size=16, common_layers=(8,))
    deep = BasicPolicy([n, n], len(gs), embedding_size=16, common_layers=(8,), policy_layers=(8,))
    pk, pn, pgs, pkw = H.config_table()["pauli3_line"]
    ppol = BasicPolicy([2 * pn, 2 * pn], len(pgs), embedding_size=16, common_layers=(8,))
    m = 65
    wide_gs = [("swap", (i, i + 1)) for i in range(m - 1)]
    wpol = BasicPolicy([m, m], len(wide_gs), embedding_size=16, common_layers=(8,))
    cfg = {"collecting": {"num_episodes": 4, "num_mcts_searches": 2}}
    with pytest.raises(NotImplementedError):
        MCTSSearch(kind, n, gs, pol, 4, 2, policy_backend="torch", use_twists=True)
    with pytest.raises(NotImplementedError):
        MCTSSearch(kind, n, gs, deep, 4, 2, use_twists=True)
    with pytest.raises(NotImplementedError):
        MCTSSearch(pk, pn, pgs, ppol, 4, 2, use_twists=True, **pkw)
    with pytest.raises(NotImplementedError):
        MCTSSearch(H.PERM, m, wide_gs, wpol, 4, 2, use_twists=True)
    with pytest.raises(ValueError):
        MCTSSearch(kind, n, gs, pol, 4, 2, use_twists=True, add_perms=False)
    with pytest.raises(NotImplementedError):
        AlphaZero(kind, n, gs, deep, cfg, use_twists=True)
    with pytest.raises(NotImplementedError):
        AlphaZero(pk, pn, pgs, ppol, cfg, use_twists=True, **pkw)
    with pytest.raises(NotImplementedError):
        AlphaZero(H.PERM, m, wide_gs, wpol, cfg, use_twists=True)
    with pytest.raises(ValueError):
        AlphaZero(kind, n, gs, pol, cfg, use_twists=True, add_perms=False)


def test_learn_keeps_each_trainers_default(monkeypatch):
    """RLSynthesis.learn(use_twists=None) builds each trainer with its own default (PPO twisted, AlphaZero untwisted); True / False are
    passed through.  The trainers are stubs: no device."""
    import qiskit_gym_b200.ppo as ppo
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    assert inspect.signature(ppo.PPO.__init__).parameters["use_twists"].default is True
    assert inspect.signature(ppo.AlphaZero.__init__).parameters["use_twists"].default is False
    made = []

    def stub(name):
        class Stub:
            def __init__(self, kind, n, gs, policy, config, **kw):
                made.append((name, kw))
                self.policy = policy

            def learn(self, **kw):
                return []
        return Stub
    monkeypatch.setattr(ppo, "PPO", stub("PPO"))
    monkeypatch.setattr(ppo, "AlphaZero", stub("AZ"))
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], max_depth=16)
    for algo in ("twisterl.rl.PPO", "twisterl.rl.AZ"):
        rls = RLSynthesis(env, {}, {"embedding_size": 16, "common_layers": [8]}, algorithm_cls=algo)
        for flag in (None, True, False):
            made.clear()
            rls.learn(num_iterations=0, use_twists=flag)
            (name, kw), = made
            assert name == algo.split(".")[-1]
            if flag is None:
                assert "use_twists" not in kw
            else:
                assert kw["use_twists"] is flag


# ---- GPU: the decisions re-enacted -------------------------------------------------------------------------------------------------
REENACT = ["C1_perm_grid3", "lf5_line_swap", "clifford3_allgates"]


def _setup(name, R, difficulty=3):
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()[name]
    kw = dict(kw, add_inverts=False)
    kw.pop("add_perms", None)
    tgt_env = orc.OracleEnv(kind, n, gs, difficulty=difficulty, add_perms=False, **kw)
    tgt_env.reset(seed=4, env_id=0)
    target = tgt_env.raw_state().astype(np.int64).tolist()
    obs_perms, act_perms = orc.OracleEnv(kind, n, gs, add_perms=True, **kw).twists()
    torch.manual_seed(1)
    probe = orc.OracleEnv(kind, n, gs, add_perms=False, **kw)
    pol = BasicPolicy(probe.obs_shape(), len(gs), embedding_size=32, common_layers=(16,))
    return kind, n, gs, kw, target, obs_perms, np.asarray(act_perms, dtype=np.int64), pol, int(np.prod(probe.obs_shape()))


def _recorder(ms):
    rec = {}
    ms.hook = lambda kind_, d, s, p, v, fr, bits: rec.__setitem__(
        (kind_, d, s), (p.cpu().numpy().copy(), None if v is None else v.cpu().numpy().copy(), fr.cpu().numpy().copy(),
                        bits.cpu().numpy().view(np.uint32).copy()))
    return rec


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("name", REENACT)
def test_twisted_tree_search_reenacted_on_cpu(name, deterministic):
    """Every evaluation's frame is k(i, e), its bits are the oracle observation of that node's env moved by obs_perms[k], the trees built
    from P = probs[act_perm[k]] give the device's root weights bit for bit, and decisions and final states match; the frames cover all K."""
    from qiskit_gym_b200.mcts import MCTSSearch
    R, S, decisions, seed, first, cp = 37, 12, 5, 21, 300, 1.5
    kind, n, gs, kw, target, obs_perms, act, pol, obs = _setup(name, R)
    A, K = len(gs), len(obs_perms)
    ekw = dict(max_depth=6, **kw)
    ms = MCTSSearch(kind, n, gs, pol, R, S, C=cp, use_twists=True, **ekw)
    assert ms.num_twists == K and K >= 2 and np.array_equal(ms.act_table.cpu().numpy(), act)
    rec = _recorder(ms)
    ms.env.set_state(target)
    ms.env.search_begin(seed, first)
    refs = []
    for b in range(R):
        r = orc.OracleEnv(kind, n, gs, add_perms=False, **ekw)
        r.set_state(target)
        refs.append(r)
    ticks = np.zeros(R, np.int64)
    chosen = torch.zeros(R, dtype=torch.int32, device=ms.env.device)
    frames, expansions = set(), 0
    for d in range(decisions):
        w_gpu = ms.decide(d).cpu().numpy()
        assert np.array_equal(ms.root_twist.cpu().numpy(), rec[("root", d, -1)][2])
        ms.env.search_step(ms.weights, deterministic=deterministic, obs=False, chosen=chosen)
        got = chosen.cpu().numpy()
        p0, _, fr0, bits0 = rec[("root", d, -1)]
        for b, r in enumerate(refs):
            g, tick = first + b, int(ticks[b])
            k = frame(seed, g, 0, tick, K)
            assert fr0[b] == k, (d, b)
            assert np.array_equal(bits0[b], _pack([obs_perms[k][i] for i in r.observe()], obs)), (d, b)
            frames.add(k)
            tree = CpuTree(r.clone(), p0[b][act[k]], A, cp)
            for s in range(S):
                p, v, fr, bits = rec[("leaf", d, s)]
                path, parent, a = tree.select()
                if a >= 0:
                    new = tree.expand(parent, a)
                    k = frame(seed, g, s + 1, tick, K)
                    assert fr[b] == k, (d, b, s)
                    assert np.array_equal(bits[b], _pack([obs_perms[k][i] for i in tree.envs[new].observe()], obs)), (d, b, s)
                    frames.add(k)
                    tree.P[new] = p[b][act[k]].astype(f32)
                    expansions += 1
                    tree.backup(path, f32(0) if tree.final[new] else v[b])
                else:
                    tree.backup(path, f32(0))
            w = tree.root_weights()
            assert np.array_equal(w.view(np.uint32), w_gpu[b].view(np.uint32)), (d, b, w, w_gpu[b])
            if r.is_final():
                assert got[b] == -1
                continue
            act_b = cpu_pick(w, orc.philox_draw(seed, g, tick, STREAM_SAMPLE), deterministic)
            assert got[b] == act_b, (d, b)
            r.step(act_b)
            ticks[b] += 1
    assert expansions > 2 * R
    assert len(frames) == K                      # the evaluations spread over the whole symmetry group
    for b in range(R):
        assert np.array_equal(ms.env.get_state(b), refs[b].raw_state())


@pytest.mark.gpu
def test_twisted_reuse_reenacted_on_cpu():
    """reuse_tree=True: re-rooted trees keep their env-order priors; fresh trees take P = probs[act_perm[k]] at k(i, 0); every leaf as above."""
    from qiskit_gym_b200.mcts import MCTSSearch
    R, S, decisions, seed, first, cp = 37, 12, 8, 21, 300, 1.5
    kind, n, gs, kw, target, obs_perms, act, pol, obs = _setup("C1_perm_grid3", R, difficulty=4)
    A, K = len(gs), len(obs_perms)
    with torch.no_grad():
        for prm in pol.action.parameters():
            prm.mul_(50.0)              # peaked priors: subtrees outgrow what a re-rooted tree keeps
    ekw = dict(max_depth=10, **kw)
    ms = MCTSSearch(kind, n, gs, pol, R, S, C=cp, reuse_tree=True, use_twists=True, **ekw)
    keep = ms.NC - S
    rec = _recorder(ms)
    ms.env.set_state(target)
    ms.env.search_begin(seed, first)
    refs = []
    for b in range(R):
        r = orc.OracleEnv(kind, n, gs, add_perms=False, **ekw)
        r.set_state(target)
        refs.append(r)
    ticks = np.zeros(R, np.int64)
    trees = [None] * R
    expected_reused = np.zeros(R, np.uint8)
    reused = 0
    for d in range(decisions):
        w_gpu = ms.decide(d).cpu().numpy()
        assert np.array_equal(ms.reused.cpu().numpy(), expected_reused), d
        ms.env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
        got = ms.chosen.cpu().numpy()
        p0, _, fr0, bits0 = rec[("root", d, -1)]
        for b, r in enumerate(refs):
            g, tick = first + b, int(ticks[b])
            k = frame(seed, g, 0, tick, K)
            assert fr0[b] == k and np.array_equal(bits0[b], _pack([obs_perms[k][i] for i in r.observe()], obs)), (d, b)
            tree = trees[b] if expected_reused[b] else ReuseTree(r.clone(), p0[b][act[k]], A, cp, b, tick, 0, False)
            for s in range(S):
                p, v, fr, bits = rec[("leaf", d, s)]
                path, parent, a = tree.select()
                if a >= 0:
                    new = tree.expand(parent, a)
                    k = frame(seed, g, s + 1, tick, K)
                    assert fr[b] == k, (d, b, s)
                    assert np.array_equal(bits[b], _pack([obs_perms[k][i] for i in tree.envs[new].observe()], obs)), (d, b, s)
                    tree.P[new] = p[b][act[k]].astype(f32)
                    tree.backup(path, f32(0) if tree.final[new] else v[b])
                else:
                    tree.backup(path, f32(0))
            w = tree.root_weights()
            assert np.array_equal(w.view(np.uint32), w_gpu[b].view(np.uint32)), (d, b)
            if r.is_final():
                assert got[b] == -1
                expected_reused[b] = 0
                continue
            act_b = cpu_pick(w, orc.philox_draw(seed, g, tick, STREAM_SAMPLE), False)
            assert got[b] == act_b, (d, b)
            r.step(act_b)
            ticks[b] += 1
            key = env_key(r, 0)
            ok = reroot(tree, act_b, lambda c: env_key(tree.envs[c], tree.inv[c]) == key, keep, NODE_FIELDS + ("envs", "tick", "inv"))
            expected_reused[b] = 1 if ok else 0
            reused += int(ok)
            trees[b] = tree
    assert reused > R
    for b in range(R):
        assert np.array_equal(ms.env.get_state(b), refs[b].raw_state())


# ---- GPU: identity table == untwisted ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("reuse", [False, True])
@pytest.mark.parametrize("name", ["C1_perm_grid3", "lf5_line_swap", "clifford3_allgates"])
def test_identity_table_equals_untwisted(name, reuse):
    """A twist table holding only the identity (K = 1) reproduces the untwisted tree search bit for bit: every decision's root weights,
    and the solutions and keys of solve, with and without reuse."""
    from qiskit_gym_b200.mcts import MCTSSearch
    R, S = 37, 12
    kind, n, gs, kw, target, _, _, pol, _ = _setup(name, R, difficulty=4)
    mk = lambda tw: MCTSSearch(kind, n, gs, pol, R, S, max_depth=10, reuse_tree=reuse, use_twists=tw, **kw)   # noqa: E731
    plain, tw = mk(False), mk(True)
    dev = tw.env.device
    tw.qperm_table = torch.arange(n, dtype=torch.uint8, device=dev).reshape(1, n)
    tw.act_table = torch.arange(tw.env.num_actions(), dtype=torch.int32, device=dev).reshape(1, -1)
    for ms in (plain, tw):
        ms.env.set_state(target)
        ms.env.search_begin(3, 11)
    for d in range(4):
        a, b = plain.decide(d).clone(), tw.decide(d).clone()
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), d
        for ms in (plain, tw):
            ms.env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
        assert torch.equal(plain.chosen, tw.chosen), d
    assert not tw.root_twist.any()
    for det in (False, True):
        for seed, first in ((1, 0), (7, 555)):
            x = plain.solve(target, deterministic=det, seed=seed, first_rollout_id=first)
            y = tw.solve(target, deterministic=det, seed=seed, first_rollout_id=first)
            assert (x.key, x.actions, x.success, x.iterations) == (y.key, y.actions, y.success, y.iterations), (det, seed, first)
            assert np.array_equal(plain.env.returns().cpu().numpy().view(np.uint32), tw.env.returns().cpu().numpy().view(np.uint32))


# ---- GPU: graph replay == eager, frames follow the seed -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sims", [12, 130])
def test_graph_replay_equals_eager(sims):
    """The captured decision (one graph up to 128 simulations, root + per-simulation graphs beyond) gives the eager search's weights,
    root and leaf frames over searches with different seeds and first ids, whose frames differ: nothing is frozen at capture."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(1)
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,))
    R = 96
    tarr = H.random_targets(kind, n, gs, R, 3, scramble=6)
    out = {}
    for graph in (False, True):
        ms = MCTSSearch(kind, n, gs, pol, R, sims, max_depth=16, add_inverts=False, use_cuda_graph=graph, use_twists=True)
        runs = []
        for seed, first in ((5, 0), (6, 0), (6, 400)):
            ms.env.set_state(tarr)
            ms.env.search_begin(seed, first)
            for d in range(3):
                w = ms.decide(d).clone()
                runs.append((w, ms.root_twist.clone(), ms.leaf_twist.clone()))
                ms.env.search_step(ms.weights, deterministic=True, obs=False)
            res = ms.solve(tarr[0].tolist(), seed=seed, first_rollout_id=first)
            runs.append((res.key, res.actions))
        out[graph] = runs
    for a, b in zip(out[False], out[True]):
        if isinstance(a[0], torch.Tensor):
            assert torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        else:
            assert a == b
    e = out[True]
    assert not torch.equal(e[0][1], e[4][1]) and not torch.equal(e[4][1], e[8][1])       # root frames follow seed and first id
    assert not torch.equal(e[0][1], e[1][1])                                               # ... and the decision's step counter


# ---- GPU: validity at K = 40 320 ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_validity_c3_all_to_all():
    """C3 (Clifford 8q, all-to-all CX: K = 40 320): every solution of the twisted tree search replays to the identity on the oracle."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, _ = H.config_table()["C3_clifford8_full"]
    kw = {"add_inverts": False}
    torch.manual_seed(1)
    pol = BasicPolicy([2 * n, 2 * n], len(gs), embedding_size=512, common_layers=(256,))
    ms = MCTSSearch(kind, n, gs, pol, 64, 16, max_depth=8, use_twists=True, **kw)
    assert ms.num_twists == 40320 and tuple(ms.act_table.shape) == (40320, len(gs))
    states = [r.tolist() for r in H.random_targets(kind, n, gs, 4, 1, scramble=1)] + [r.tolist() for r in H.random_targets(kind, n, gs, 4, 2, scramble=2)]
    solved = 0
    for t, st in enumerate(states):
        res = ms.solve(st, seed=17 + t)
        if res.success:
            solved += 1
            assert _replays_to_success(kind, n, gs, kw, st, res.actions, max_depth=8), t
    assert solved >= 4
    assert len(set(ms.root_twist.cpu().tolist())) > 30


# ---- GPU: AlphaZero ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_alphazero_twisted_samples():
    """One twisted self-play: each sample's observation is the unpacked twisted root bits of its decision, its target the root weights
    scattered through act_perm[k] (policy order); the env played the env-order weights."""
    from qiskit_gym_b200.collector import unpack_bits
    from qiskit_gym_b200.ppo import AlphaZero
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=32, common_layers=(32,))
    cfg = {"collecting": {"num_episodes": 64, "num_mcts_searches": 8, "C": 1.41}, "training": {"num_epochs": 1}}
    az = AlphaZero(kind, n, gs, pol, cfg, device=0, seed=3, use_twists=True, add_inverts=False)
    ms = az.search
    assert ms.use_twists and ms.num_twists == 8
    seen = []
    decide = ms.decide

    def recording(d=0):
        w = decide(d)
        seen.append((ms.root_bits.clone(), ms.root_twist.clone(), w.clone()))
        return w
    ms.decide = recording
    az.difficulty = 3
    _, obs, tgt_pi, _, idx = az.self_play()
    B, A = ms.R, ms.env.num_actions()
    all_obs = torch.stack([unpack_bits(b, ms.env._obs_size).reshape(B, n, n) for b, _, _ in seen]).reshape(-1, n, n)
    all_pi = torch.zeros((len(seen), B, A), device=obs.device)
    act = ms.act_table.cpu().numpy()
    for t, (_, k, w) in enumerate(seen):
        kk, ww = k.cpu().numpy(), w.cpu().numpy()
        ref = np.zeros((B, A), np.float32)
        for i in range(B):
            ref[i, act[kk[i]]] = ww[i]
        all_pi[t] = torch.from_numpy(ref)
    assert len(set(torch.cat([k for _, k, _ in seen]).tolist())) == 8
    assert idx.numel() > B
    assert torch.equal(obs, all_obs.reshape(-1, n, n)[idx])
    assert torch.equal(tgt_pi.view(torch.int32), all_pi.reshape(-1, A)[idx].view(torch.int32))


@pytest.mark.gpu
def test_alphazero_learns_permutation_line4_twisted():
    """The budget of test_ppo.py::test_alphazero_learns_permutation_line4 with learn(use_twists=True): the curriculum reaches difficulty 3
    with finite losses."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    torch.manual_seed(0)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], difficulty=1, depth_slope=2, max_depth=32)
    cfg = {"collecting": {"num_episodes": 256, "num_mcts_searches": 16, "C": 1.41}, "training": {"num_epochs": 4}, "optimizer": {"lr": 2e-3},
           "learning": {"diff_threshold": 0.85, "diff_max": 6, "diff_metric": "mcts_16"},
           "evals": {"ppo_deterministic": {"num_episodes": 64}, "mcts_16": {"num_episodes": 64, "num_mcts_searches": 16}}}
    rls = RLSynthesis(env, cfg, {"embedding_size": 64, "common_layers": [64]}, device=0, algorithm_cls="twisterl.rl.AZ")
    hist = rls.learn(initial_difficulty=1, num_iterations=25, use_twists=True)
    trace = [(h["difficulty"], round(h["eval/mcts_16"], 2), round(h["eval/ppo_deterministic"], 2)) for h in hist]
    assert hist[-1]["difficulty"] >= 3, trace
    assert all(np.isfinite(h["loss"]) for h in hist)
