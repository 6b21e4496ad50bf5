"""The tree search on the tensor-core policy (MCTSSearch(policy_backend="tensor_core")), AlphaZero self-play on it (AlphaZero(matmul_precision=
"tensor_core")) and RLSynthesis.solve / synth(matmul_precision="tensor_core").

The backend changes only where the priors and values come from: qg_policy_tc_forward_bits on the packed bits the search already produces
(env.observe_bits for the roots, qg_step_slots for the leaves, qg_mcts_observe_twisted when twisted).  So the trees are re-enacted on the
CPU (tests/test_mcts.py::CpuTree and the twisted / reuse restatements) from the outputs the device trees consumed, and those outputs are
checked against the float64 module within TensorCorePolicy's bound (tests/test_policy_tc_envelope.py::Refs).

Row independence.  Every random draw of a tree search is keyed by the rollout's global id or the tree's index, never by the launch width
(csrc/qg_mcts.cu, csrc/qg_kernels.cuh): the decision's sample is philox(seed; first_id + i, tick, STREAM_SAMPLE); a node's add_inverts coin
is drawn by the slot pool's step from (pool seed, pool first id + i, the parent's step counter), i being the tree's logical index in
qg_step_slots; a twisted evaluation's frame is philox(seed; first_id + i + (e << 32), tick, STREAM_TWIST).  The tree kernels are one warp
per tree with no cross-tree communication.  With TensorCorePolicy's rows bit-identical whatever the batch, tree i of an R-tree search
therefore equals tree i of an R'-tree search on the same targets."""
import inspect

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_mcts import CpuTree
from tests.test_mcts_reuse import NODE_FIELDS, ReuseTree, env_key, reroot
from tests.test_mcts_twist import _pack, frame
from tests.test_policy_tc_envelope import Refs
from tests.test_search import STREAM_SAMPLE, cpu_pick
from tests.test_search_many import _replays_to_success

f32 = np.float32


# ---- CPU: refusals before any allocation, defaults -----------------------------------------------------------------------------------
def _no_engine(monkeypatch):
    import qiskit_gym_b200.mcts as mcts
    import qiskit_gym_b200.ppo as ppo
    import qiskit_gym_b200.search as search

    def refuse(*a, **k):
        raise AssertionError("an engine was allocated before the refusal")
    for mod in (mcts, ppo, search):
        monkeypatch.setattr(mod, "BatchedEnv", refuse)


def _refusal_cases():
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, _ = H.config_table()["C1_perm_grid3"]
    pol = BasicPolicy([n, n], len(gs), embedding_size=16, common_layers=(8,))
    deep = BasicPolicy([n, n], len(gs), embedding_size=16, common_layers=(8,), value_layers=(8,))
    m = 17                                            # 136 SWAP actions: more than the tensor-core head's 127 (+ the value column)
    many_gs = [("swap", (i, j)) for i in range(m) for j in range(i + 1, m)]
    many = BasicPolicy([m, m], len(many_gs), embedding_size=16, common_layers=(8,))
    w = 65                                            # no packed observations past 64 qubits
    wide_gs = [("swap", (i, i + 1)) for i in range(w - 1)]
    wide = BasicPolicy([w, w], len(wide_gs), embedding_size=16, common_layers=(8,))
    return (kind, n, gs, pol), [(kind, n, gs, deep), (H.PERM, m, many_gs, many), (H.PERM, w, wide_gs, wide)]


def test_refusals_before_any_device_work(monkeypatch):
    """MCTSSearch(policy_backend="tensor_core") and AlphaZero(matmul_precision="tensor_core") refuse a policy without single-Linear heads,
    more than 127 actions and a Permutation wider than 64 qubits (NotImplementedError), twisted or not, before any engine; AlphaZero refuses
    an unknown precision (ValueError)."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.ppo import AlphaZero
    _no_engine(monkeypatch)
    (kind, n, gs, pol), bad = _refusal_cases()
    cfg = {"collecting": {"num_episodes": 4, "num_mcts_searches": 2}}
    for k, m, g, p in bad:
        for tw in (False, True):
            with pytest.raises(NotImplementedError):
                MCTSSearch(k, m, g, p, 4, 2, policy_backend="tensor_core", use_twists=tw)
            with pytest.raises(NotImplementedError):
                AlphaZero(k, m, g, p, cfg, matmul_precision="tensor_core", use_twists=tw)
    for prec in ("tf32", "bf16", "fp8"):
        with pytest.raises(ValueError):
            AlphaZero(kind, n, gs, pol, cfg, matmul_precision=prec)


def test_refuses_a_device_that_is_not_sm100(monkeypatch):
    """The sm_100 check fires before any engine (the device is asked, not used)."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.ppo import AlphaZero
    _no_engine(monkeypatch)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "get_device_capability", lambda device=None: (9, 0))
    (kind, n, gs, pol), _ = _refusal_cases()
    with pytest.raises(NotImplementedError):
        MCTSSearch(kind, n, gs, pol, 4, 2, policy_backend="tensor_core")
    with pytest.raises(NotImplementedError):
        AlphaZero(kind, n, gs, pol, {"collecting": {"num_episodes": 4, "num_mcts_searches": 2}}, matmul_precision="tensor_core")


def test_rlsynthesis_refusals(monkeypatch):
    """solve / synth(matmul_precision=...): an unknown precision is a ValueError, the tensor-core limits NotImplementedError, for the tree
    and the rollout search; the refusals that existed stay; learn() with AZ still refuses tf32 / bf16 and update_precision="tensor_core".
    No engine is allocated."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    _no_engine(monkeypatch)
    m = 17
    spec = SynthSpec.from_coupling_map("PermutationEnv", [(i, j) for i in range(m) for j in range(i + 1, m)], max_depth=8)
    rls = RLSynthesis(spec, {}, {"embedding_size": 16, "common_layers": [8]})
    for sims in (0, 2):
        with pytest.raises(NotImplementedError):
            rls.solve(list(range(m)), num_searches=4, num_mcts_searches=sims, matmul_precision="tensor_core")
        with pytest.raises(NotImplementedError):
            rls.synth(list(range(m)), num_searches=4, num_mcts_searches=sims, matmul_precision="tensor_core")
        with pytest.raises(ValueError):
            rls.solve(list(range(m)), num_searches=4, num_mcts_searches=sims, matmul_precision="bf16")
    small = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2)], max_depth=8)
    rls = RLSynthesis(small, {}, {"embedding_size": 16, "common_layers": [8]})
    with pytest.raises(NotImplementedError):
        rls.solve([0, 1, 2], num_searches=4, num_mcts_searches=2, use_twists=True, matmul_precision="tensor_core")
    with pytest.raises(NotImplementedError):
        rls.solve([0, 1, 2], num_searches=4, num_mcts_searches=2, max_expand_depth=2, matmul_precision="tensor_core")
    with pytest.raises(NotImplementedError):
        rls.solve_many([[0, 1, 2]], num_searches=4, num_mcts_searches=2, matmul_precision="tensor_core")
    with pytest.raises(NotImplementedError):
        rls.synth_many([[0, 1, 2]], num_searches=4, num_mcts_searches=2, matmul_precision="tensor_core")
    deep = RLSynthesis(small, {}, {"embedding_size": 16, "common_layers": [8], "value_layers": [8]})
    with pytest.raises(NotImplementedError):
        deep.solve([0, 1, 2], num_searches=4, num_mcts_searches=2, matmul_precision="tensor_core")
    rls.algorithm_cls = "twisterl.rl.AZ"
    for prec in ("tf32", "bf16"):
        with pytest.raises(NotImplementedError):
            rls.learn(num_iterations=1, matmul_precision=prec)
    with pytest.raises(NotImplementedError):
        rls.learn(num_iterations=1, matmul_precision="tensor_core", update_precision="tensor_core")


def test_defaults_and_learn_pass_through(monkeypatch):
    """The defaults stay f32 / "auto", and learn(matmul_precision="tensor_core") reaches the AlphaZero trainer (a stub: no device)."""
    import qiskit_gym_b200.ppo as ppo
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    assert inspect.signature(MCTSSearch.__init__).parameters["policy_backend"].default == "auto"
    assert inspect.signature(ppo.AlphaZero.__init__).parameters["matmul_precision"].default == "f32"
    for fn in (RLSynthesis.solve, RLSynthesis.synth, RLSynthesis.learn):
        assert inspect.signature(fn).parameters["matmul_precision"].default == "f32"
    made = []

    class Stub:
        def __init__(self, kind, n, gs, policy, config, **kw):
            made.append(kw)
            self.policy = policy

        def learn(self, **kw):
            return []
    monkeypatch.setattr(ppo, "AlphaZero", Stub)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], max_depth=16)
    rls = RLSynthesis(env, {}, {"embedding_size": 16, "common_layers": [8]}, algorithm_cls="twisterl.rl.AZ")
    for prec in ("f32", "tensor_core"):
        made.clear()
        rls.learn(num_iterations=0, matmul_precision=prec)
        (kw,) = made
        assert kw["matmul_precision"] == prec and "update_precision" not in kw


# ---- GPU: the decisions re-enacted, the outputs within the bound ----------------------------------------------------------------------
REENACT = [("C1_perm_grid3", False), ("C1_perm_grid3", True), ("lf5_line_swap", False), ("lf5_line_swap", True),
           ("clifford3_allgates", False), ("clifford3_allgates", True), ("pauli3_line", False), ("pauli3_line", True)]


def _reenact(name, deterministic, twisted=False, reuse=False):
    """Decisions of a "tensor_core" tree search re-enacted on the CPU from the priors and values its trees consumed (recorded by the hook):
    root weights bit for bit, decisions, re-rooting, frames and observation bits (twisted), final states.  Then every evaluation's outputs
    (root priors; leaf priors and values) against the float64 module on the evaluation's own observation, within TensorCorePolicy's bound."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.policy import TensorCorePolicy
    from qiskit_gym_b200.search import BasicPolicy
    R, S, seed, first, cp = 37, 12, 21, 300, 1.5
    decisions = 8 if reuse else 5
    kind, n, gs, kw = H.config_table()[name]
    kw = dict(kw)
    kw.pop("add_perms", None)
    if kind != H.PAULI:
        kw["add_inverts"] = False
    if kind == H.PAULI:
        t = H.random_targets(kind, n, gs, 1, 3, scramble=3, num_rotations=2)
        target = t[0, : H.payload_lengths(kind, n, t)[0]].tolist()
    else:
        e = orc.OracleEnv(kind, n, gs, difficulty=4 if reuse else 3, add_perms=False, **kw)
        e.reset(seed=4, env_id=0)
        target = e.raw_state().astype(np.int64).tolist()
    ekw = dict(max_depth=10 if reuse else 6, **kw)
    probe = orc.OracleEnv(kind, n, gs, add_perms=False, **ekw)
    obs, A = int(np.prod(probe.obs_shape())), len(gs)
    torch.manual_seed(1)
    pol = BasicPolicy(probe.obs_shape(), A, embedding_size=32, common_layers=(16,))
    if reuse:
        with torch.no_grad():
            for prm in pol.action.parameters():
                prm.mul_(50.0)          # peaked priors: subtrees outgrow what a re-rooted tree keeps
    if twisted:
        obs_perms, act = orc.OracleEnv(kind, n, gs, add_perms=True, **kw).twists()
        act = np.asarray(act, dtype=np.int64)
    else:
        obs_perms, act = [np.arange(obs)], np.arange(A, dtype=np.int64)[None, :]
    K = len(obs_perms)
    ms = MCTSSearch(kind, n, gs, pol, R, S, C=cp, policy_backend="tensor_core", reuse_tree=reuse, use_twists=twisted, **ekw)
    assert ms.backend == "tensor_core" and isinstance(ms.handle, TensorCorePolicy) and ms.fused is None and ms.handle.max_batch == R
    if twisted:
        assert ms.num_twists == K and np.array_equal(ms.act_table.cpu().numpy(), act)
    keep = ms.NC - S
    rec = {}
    ms.hook = lambda kind_, d, s, p, v, *tw: rec.__setitem__(
        (kind_, d, s), (p.cpu().numpy().copy(), None if v is None else v.cpu().numpy().copy(), *[x.cpu().numpy().copy() for x in tw]))
    ms.env.set_state(target)
    ms.env.search_begin(seed, first)
    refs = []
    for b in range(R):
        r = orc.OracleEnv(kind, n, gs, add_perms=False, **ekw)
        r.set_state(target)
        refs.append(r)
    ticks = np.zeros(R, np.int64)
    trees, expected_reused = [None] * R, np.zeros(R, np.uint8)
    roots, leaves = ([], []), ([], [], [])            # (observation indices, priors[, values]) of every evaluation the trees consumed
    expansions = reused = 0
    for d in range(decisions):
        w_gpu = ms.decide(d).cpu().numpy()
        if reuse:
            assert np.array_equal(ms.reused.cpu().numpy(), expected_reused), d
        ms.env.search_step(ms.weights, deterministic=deterministic, obs=False, chosen=ms.chosen)
        got = ms.chosen.cpu().numpy()
        p0, _, *tw0 = rec[("root", d, -1)]
        for b, r in enumerate(refs):
            g, tick = first + b, int(ticks[b])
            k = frame(seed, g, 0, tick, K) if twisted else 0
            idx = [int(obs_perms[k][i]) for i in r.observe()]
            if twisted:
                assert tw0[0][b] == k and np.array_equal(tw0[1][b].view(np.uint32), _pack(idx, obs)), (d, b)
            roots[0].append(idx)
            roots[1].append(p0[b])
            if expected_reused[b]:
                tree = trees[b]
            elif reuse:
                tree = ReuseTree(r.clone(), p0[b][act[k]], A, cp, b, tick, 0, False)
            else:
                tree = CpuTree(r.clone(), p0[b][act[k]], A, cp)
            for s in range(S):
                p, v, *tw = rec[("leaf", d, s)]
                path, parent, a = tree.select()
                if a >= 0:
                    new = tree.expand(parent, a)
                    k = frame(seed, g, s + 1, tick, K) if twisted else 0
                    idx = [int(obs_perms[k][i]) for i in tree.envs[new].observe()]
                    if twisted:
                        assert tw[0][b] == k and np.array_equal(tw[1][b].view(np.uint32), _pack(idx, obs)), (d, b, s)
                    tree.P[new] = p[b][act[k]].astype(f32)
                    for lst, x in zip(leaves, (idx, p[b], v[b])):
                        lst.append(x)
                    expansions += 1
                    tree.backup(path, f32(0) if tree.final[new] else v[b])
                else:
                    tree.backup(path, f32(0))
            w = tree.root_weights()
            assert np.array_equal(w.view(np.uint32), w_gpu[b].view(np.uint32)), (d, b, w, w_gpu[b])
            if r.is_final():
                assert got[b] == -1
                expected_reused[b] = 0
                continue
            act_b = cpu_pick(w, orc.philox_draw(seed, g, tick, STREAM_SAMPLE), deterministic)
            assert got[b] == act_b, (d, b)
            r.step(act_b)
            ticks[b] += 1
            if reuse:
                key = env_key(r, 0)
                ok = reroot(tree, act_b, lambda c: env_key(tree.envs[c], tree.inv[c]) == key, keep, NODE_FIELDS + ("envs", "tick", "inv"))
                expected_reused[b] = 1 if ok else 0
                reused += int(ok)
                trees[b] = tree
    assert expansions > 2 * R                         # trees really grew
    if reuse:
        assert reused > R
    for b in range(R):
        assert np.array_equal(ms.env.get_state(b), refs[b].raw_state())
    dev = ms.env.device

    def dense(rows):
        x = np.zeros((len(rows), obs), np.float32)
        for i, idx in enumerate(rows):
            x[i, idx] = 1.0
        return torch.from_numpy(x).to(dev)
    Refs(ms.policy, dense(roots[0]), with_value=True).check(len(roots[0]), probs=torch.from_numpy(np.stack(roots[1])).to(dev), tag="roots")
    Refs(ms.policy, dense(leaves[0]), with_value=True).check(len(leaves[0]), probs=torch.from_numpy(np.stack(leaves[1])).to(dev),
                                                             values=torch.from_numpy(np.asarray(leaves[2], np.float32)).to(dev), tag="leaves")


@pytest.mark.gpu
@pytest.mark.parametrize("name,deterministic", REENACT)
def test_reenacted_on_cpu(name, deterministic):
    _reenact(name, deterministic)


@pytest.mark.gpu
@pytest.mark.parametrize("name,deterministic", [(nm, d) for nm, d in REENACT if nm != "pauli3_line"])
def test_twisted_reenacted_on_cpu(name, deterministic):
    _reenact(name, deterministic, twisted=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name,twisted", [("C1_perm_grid3", False), ("lf5_line_swap", False), ("C1_perm_grid3", True)])
def test_reuse_reenacted_on_cpu(name, twisted):
    _reenact(name, False, twisted=twisted, reuse=True)


# ---- GPU: a tree does not depend on how many trees share the launch ----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
def test_tree_independent_of_launch_width(twisted):
    """Tree i of R-tree "tensor_core" searches on the same per-rollout targets, R = 1, 127, 128, 129 (both sides of a 128-row tile) and
    1 184: the same root weights bit for bit at every decision, the same decisions and returns (module docstring: why this must hold).
    add_inverts is on, so the pool's coins are part of what must not depend on R."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    kw = dict(kw, add_inverts=True)
    torch.manual_seed(2)
    pol = BasicPolicy([n, n], len(gs), embedding_size=128, common_layers=(64,))
    Rs = (1184, 1, 127, 128, 129)
    tarr = H.random_targets(kind, n, gs, max(Rs), 3, scramble=8)
    out = {}
    for R in Rs:
        ms = MCTSSearch(kind, n, gs, pol, R, 16, max_depth=12, policy_backend="tensor_core", use_twists=twisted, **kw)
        ms.env.set_state(tarr[:R])
        ms.env.search_begin(9, 40)
        runs = []
        for d in range(6):
            w = ms.decide(d).clone()
            ms.env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
            runs.append((w.view(torch.int32), ms.chosen.clone()))
        out[R] = (runs, ms.env.returns().clone().view(torch.int32))
        del ms
    ref_runs, ref_ret = out[1184]
    assert any(bool((c >= 0).any()) for _, c in ref_runs[1:])
    for R in Rs[1:]:
        runs, ret = out[R]
        for d, ((w, c), (rw, rc)) in enumerate(zip(runs, ref_runs)):
            assert torch.equal(w, rw[:R]) and torch.equal(c, rc[:R]), (R, d)
        assert torch.equal(ret, ref_ret[:R]), R


# ---- GPU: graphs, refresh ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
@pytest.mark.parametrize("sims", [12, 130])
def test_graph_replay_equals_eager(sims, twisted):
    """The captured decision (one graph up to 128 simulations, root + per-simulation graphs beyond) gives the launch-by-launch search's
    weights bit for bit over searches with different seeds and first ids, and the same solve results."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(1)
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,))
    R = 96
    tarr = H.random_targets(kind, n, gs, R, 3, scramble=6)
    out = {}
    for graph in (False, True):
        ms = MCTSSearch(kind, n, gs, pol, R, sims, max_depth=16, add_inverts=False, use_cuda_graph=graph, policy_backend="tensor_core",
                        use_twists=twisted)
        runs = []
        for seed, first in ((5, 0), (6, 400)):
            ms.env.set_state(tarr)
            ms.env.search_begin(seed, first)
            for d in range(3):
                runs.append(ms.decide(d).clone().view(torch.int32))
                ms.env.search_step(ms.weights, deterministic=True, obs=False)
            res = ms.solve(tarr[0].tolist(), seed=seed, first_rollout_id=first)
            runs.append((res.key, res.actions))
        assert (ms._graphs is not None) == graph
        out[graph] = runs
    for a, b in zip(out[False], out[True]):
        assert torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b


def _decisions(ms, tarr, seed=5):
    """Root weights of 3 decisions, then the priors and values of the last leaf evaluation (as int32 bits)."""
    ms.env.set_state(tarr)
    ms.env.search_begin(seed, 0)
    ms.chosen.fill_(-1)
    ms._fresh = True
    out = []
    for d in range(3):
        out.append(ms.decide(d).clone().view(torch.int32))
        ms.env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
    return out + [ms.pri.clone().view(torch.int32), ms.val.clone().view(torch.int32)]


@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
def test_in_place_refresh_keeps_the_graphs(twisted):
    """After an optimiser step on the module, and after load_state_dict, the next decisions equal those of a freshly built "tensor_core"
    search on the new weights, replayed by the graphs captured before the update (the handle loaded the weights in place)."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(3)
    pol = BasicPolicy([n, n], len(gs), embedding_size=128, common_layers=(64,))
    other = BasicPolicy([n, n], len(gs), embedding_size=128, common_layers=(64,))
    R, S = 200, 48
    tarr = H.random_targets(kind, n, gs, R, 3, scramble=6)
    mk = lambda: MCTSSearch(kind, n, gs, pol, R, S, max_depth=16, add_inverts=False, policy_backend="tensor_core", use_twists=twisted)  # noqa: E731
    ms = mk()
    before = _decisions(ms, tarr)
    graph, handle = ms._graphs[3], ms.handle._h
    assert graph is not None
    opt = torch.optim.Adam(pol.parameters(), lr=0.05)
    x = (torch.rand((64, n, n), device=ms.env.device) < 0.5).float()
    logits, value = pol(x)
    (logits.logsumexp(-1).mean() + value.square().mean()).backward()
    opt.step()
    stepped = _decisions(ms, tarr)
    assert ms._graphs[3] is graph and ms.handle._h is handle
    assert not torch.equal(before[-2], stepped[-2]) and any(not torch.equal(a, b) for a, b in zip(before[:3], stepped[:3]))
    fresh = _decisions(mk(), tarr)
    assert all(torch.equal(a, b) for a, b in zip(stepped, fresh))
    pol.load_state_dict(other.state_dict())
    loaded = _decisions(ms, tarr)
    assert ms._graphs[3] is graph and ms.handle._h is handle
    fresh = _decisions(mk(), tarr)
    assert all(torch.equal(a, b) for a, b in zip(loaded, fresh))


# ---- GPU: validity at scale ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
def test_validity_c3_4096_trees(twisted):
    """C3 (Clifford 8q, all-to-all CX) with the default-shape policy (256 -> 512 -> 256 -> A + 1), 4 096 trees x 16 simulations: every
    returned solution replays to the identity on the oracle."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, _ = H.config_table()["C3_clifford8_full"]
    kw = {"add_inverts": False}
    torch.manual_seed(1)
    pol = BasicPolicy([2 * n, 2 * n], len(gs), embedding_size=512, common_layers=(256,))
    ms = MCTSSearch(kind, n, gs, pol, 4096, 16, max_depth=8, policy_backend="tensor_core", use_twists=twisted, **kw)
    states = [r.tolist() for r in H.random_targets(kind, n, gs, 4, 1, scramble=1)] + [r.tolist() for r in H.random_targets(kind, n, gs, 4, 2, scramble=2)]
    solved = 0
    for t, st in enumerate(states):
        res = ms.solve(st, seed=17 + t)
        assert res.rollouts == 4096
        if res.success:
            solved += 1
            assert _replays_to_success(kind, n, gs, kw, st, res.actions, max_depth=8), t
    assert solved >= 2                  # (a random-weight policy: the count only guards against a search that never succeeds)


# ---- GPU: AlphaZero, RLSynthesis ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
def test_alphazero_samples(twisted):
    """One self-play on the tensor-core tree search: each sample's observation is its decision's unpacked root bits, its target the root
    weights (scattered through act_perm[k] when twisted); the evals keep the f32 ("fused") tree search."""
    from qiskit_gym_b200.collector import unpack_bits
    from qiskit_gym_b200.ppo import AlphaZero
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=32, common_layers=(32,))
    cfg = {"collecting": {"num_episodes": 64, "num_mcts_searches": 8, "C": 1.41}, "training": {"num_epochs": 1},
           "evals": {"mcts_4": {"num_episodes": 16, "num_mcts_searches": 4}}, "learning": {"diff_metric": "mcts_4"}}
    az = AlphaZero(kind, n, gs, pol, cfg, device=0, seed=3, use_twists=twisted, matmul_precision="tensor_core", add_inverts=False)
    ms = az.search
    assert ms.backend == "tensor_core" and ms.use_twists == twisted
    seen = []
    decide = ms.decide

    def recording(d=0):
        w = decide(d)
        seen.append((ms.root_bits.clone(), ms.root_twist.clone() if twisted else None, w.clone()))
        return w
    ms.decide = recording
    az.difficulty = 3
    _, obs, tgt_pi, _, idx = az.self_play()
    B, A = ms.R, ms.env.num_actions()
    all_obs = torch.stack([unpack_bits(b, ms.env._obs_size).reshape(B, n, n) for b, _, _ in seen]).reshape(-1, n, n)
    all_pi = torch.zeros((len(seen), B, A), device=obs.device)
    for t, (_, k, w) in enumerate(seen):
        if not twisted:
            all_pi[t] = w
            continue
        act, kk, ww = ms.act_table.cpu().numpy(), k.cpu().numpy(), w.cpu().numpy()
        ref = np.zeros((B, A), np.float32)
        for i in range(B):
            ref[i, act[kk[i]]] = ww[i]
        all_pi[t] = torch.from_numpy(ref)
    assert idx.numel() > B
    assert torch.equal(obs, all_obs.reshape(-1, n, n)[idx])
    assert torch.equal(tgt_pi.view(torch.int32), all_pi.reshape(-1, A)[idx].view(torch.int32))
    az.evaluate("mcts_4")
    assert [m.backend for m in az._eval_mcts.values()] == ["fused"]


@pytest.mark.gpu
def test_defaults_unchanged_on_device():
    """MCTSSearch without policy_backend and AlphaZero without matmul_precision build the f32 fused tree search as before."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.policy import FusedPolicy
    from qiskit_gym_b200.ppo import AlphaZero
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    pol = BasicPolicy([n, n], len(gs), embedding_size=32, common_layers=(32,))
    ms = MCTSSearch(kind, n, gs, pol, 8, 4, **kw)
    assert ms.backend == "fused" and isinstance(ms.handle, FusedPolicy) and ms.fused is ms.handle
    az = AlphaZero(kind, n, gs, pol, {"collecting": {"num_episodes": 8, "num_mcts_searches": 4}}, device=0, **kw)
    assert az.search.backend == "fused"


@pytest.mark.gpu
@pytest.mark.parametrize("twisted", [False, True])
def test_alphazero_tensor_core_learns_permutation_line4(twisted):
    """The budget of tests/test_ppo.py::test_alphazero_learns_permutation_line4 (the env, config, seeds and iterations of
    RLSynthesis.learn) with self-play on the tensor-core tree search: the curriculum reaches difficulty 3 with finite losses."""
    from qiskit_gym_b200.ppo import AlphaZero
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    torch.manual_seed(0)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], difficulty=1, depth_slope=2, max_depth=32)
    cfg = {"collecting": {"num_episodes": 256, "num_mcts_searches": 16, "C": 1.41}, "training": {"num_epochs": 4}, "optimizer": {"lr": 2e-3},
           "learning": {"diff_threshold": 0.85, "diff_max": 6, "diff_metric": "mcts_16"},
           "evals": {"ppo_deterministic": {"num_episodes": 64}, "mcts_16": {"num_episodes": 64, "num_mcts_searches": 16}}}
    rls = RLSynthesis(env, cfg, {"embedding_size": 64, "common_layers": [64]}, device=0, algorithm_cls="twisterl.rl.AZ")
    kind, n, gs, kw = rls._env_args()
    az = AlphaZero(kind, n, gs, rls.policy, rls.rl_config, device=0, seed=0, matmul_precision="tensor_core", use_twists=twisted, **kw)
    assert az.search.backend == "tensor_core"
    hist = az.learn(initial_difficulty=1, num_iterations=25)
    trace = [(h["difficulty"], round(h["eval/mcts_16"], 2), round(h["eval/ppo_deterministic"], 2)) for h in hist]
    assert hist[-1]["difficulty"] >= 3, trace
    assert all(np.isfinite(h["loss"]) for h in hist)


@pytest.mark.gpu
def test_rlsynthesis_solve_tensor_core():
    """solve(matmul_precision="tensor_core"): the tree search is MCTSSearch's "tensor_core" backend, cached beside the f32 one, and
    returns what such a search returns; without tree search it is the "tensor_core" rollout search."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.search import RolloutSearch
    from qiskit_gym_b200.specs import SynthSpec
    torch.manual_seed(0)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3), (3, 4)], difficulty=3, max_depth=16)
    rls = RLSynthesis(env, {}, {"embedding_size": 64, "common_layers": [64]}, device=0)
    kind, n, gs, kw = rls._env_args(add_perms=False)
    states = [[1, 0, 2, 3, 4], [0, 2, 1, 4, 3], [4, 3, 2, 1, 0]]
    ref_tree = MCTSSearch(kind, n, gs, rls.policy, 32, 8, C=1.41, device=0, policy_backend="tensor_core", **kw)
    ref_roll = RolloutSearch(kind, n, gs, rls.policy, 32, device=0, policy_backend="tensor_core", **kw)
    for st in states:
        assert rls.solve(st, num_searches=32, num_mcts_searches=8, C=1.41, seed=2, matmul_precision="tensor_core") == \
            ref_tree.solve(st, seed=2).actions
        assert rls.solve(st, num_searches=32, seed=2, matmul_precision="tensor_core") == ref_roll.solve(st, seed=2).actions
        rls.solve(st, num_searches=32, num_mcts_searches=8, C=1.41, seed=2)
    tc = rls._searches[("tensor_core", ("mcts", 32, 8, 1.41, False))]
    assert tc.backend == "tensor_core" and rls._searches[("mcts", 32, 8, 1.41, False)].backend == "fused"
    assert rls._searches[("tensor_core", 32)].backend == "tensor_core"
