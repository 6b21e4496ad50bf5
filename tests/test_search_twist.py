"""The twisted rollout search (RolloutSearch(use_twists=True), RLSynthesis.solve / synth / solve_many / synth_many(use_twists=True)): every
rollout runs the policy in a symmetry frame of the env drawn per decision, k = mulhi(philox(seed; g, tick, 5), K).  Its decisions are re-enacted
on the CPU with the oracle envs and the oracle's twists; the one-launch search equals the two-launch one bit for bit; a table holding only
the identity reproduces the untwisted search; solve_many keeps its contract; solutions at K = 40 320 are valid; the refusals need no device."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_search import STREAM_SAMPLE, cpu_pick, order_key
from tests.test_search_many import MAX_DEPTH, _config, _policy, _replays_to_success, _same, _targets

STREAM_TWIST = 5


def twist_index(seed, g, tick, K):
    return (orc.philox_draw(seed, g, tick, STREAM_TWIST) * K) >> 32


def _pack(indices, obs):
    bits = np.zeros((obs + 31) // 32 * 32, dtype=np.uint8)
    bits[list(indices)] = 1
    return np.packbits(bits, bitorder="little").view(np.uint32)


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_refusals_before_any_device_work():
    """The "torch" backend, PauliNetwork, a Permutation wider than 64 qubits and the tree search refuse use_twists up front."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch, check_twisted_search
    from qiskit_gym_b200.specs import SynthSpec
    kind, n, gs, _ = H.config_table()["C1_perm_grid3"]
    pol = BasicPolicy([n, n], len(gs), embedding_size=16, common_layers=(8,))
    with pytest.raises(NotImplementedError):
        RolloutSearch(kind, n, gs, pol, 4, policy_backend="torch", use_twists=True)
    pk, pn, pgs, pkw = H.config_table()["pauli3_line"]
    for backend in ("persistent", "fused", "tensor_core"):
        with pytest.raises(NotImplementedError):
            RolloutSearch(pk, pn, pgs, pol, 4, policy_backend=backend, use_twists=True, **pkw)
    with pytest.raises(NotImplementedError):
        check_twisted_search(H.PERM, 65, "persistent")
    check_twisted_search(H.PERM, 64, "persistent")
    check_twisted_search(H.CLIFF, 8, "tensor_core")
    with pytest.raises(ValueError):
        RolloutSearch(kind, n, gs, pol, 4, use_twists=True, add_perms=False)

    grid = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (0, 3), (1, 4), (2, 5), (3, 4), (4, 5)], max_depth=8)
    rls = RLSynthesis(grid, {}, {"embedding_size": 16, "common_layers": [8]})
    with pytest.raises(NotImplementedError):
        rls.solve(list(range(6)), num_searches=4, num_mcts_searches=2, use_twists=True)
    with pytest.raises(NotImplementedError):
        rls.synth([("swap", (0, 1))], num_searches=4, num_mcts_searches=2, use_twists=True)
    with pytest.raises(NotImplementedError):
        rls.solve_many([list(range(6))], num_searches=4, num_mcts_searches=2, use_twists=True)
    m = 65
    wide = SynthSpec.from_coupling_map("PermutationEnv", [(i, i + 1) for i in range(m - 1)], max_depth=8)
    rw = RLSynthesis(wide, {}, {"embedding_size": 16, "common_layers": [8]})
    with pytest.raises(NotImplementedError):
        rw.solve(list(range(m)), num_searches=4, use_twists=True)
    with pytest.raises(NotImplementedError):
        rw.synth_many([list(range(m))], num_searches=4, use_twists=True)
    tri = [(0, 1), (1, 0), (1, 2), (2, 1)]
    pauli = SynthSpec.from_coupling_map("PauliNetworkEnv", tri, basis_gates=("H", "S", "SX", "CX"), max_depth=16)
    rp = RLSynthesis(pauli, {}, {"embedding_size": 16, "common_layers": [8]})
    with pytest.raises(NotImplementedError):
        rp.synth_many([([], ["ZZI"])], num_searches=4, use_twists=True)
    assert rls._searches == {} and rw._searches == {} and rp._searches == {}


def test_twist_tables_are_qubit_lifts():
    """The tables the twisted search keeps come from the engine's twists (collector.qubit_twist_table): on the oracle's obs perms of C1
    (3x3 grid, K = 8), lifting each inverse qubit permutation gives back the obs perm."""
    from qiskit_gym_b200.collector import qubit_twist_table
    kind, n, gs, _ = H.config_table()["C1_perm_grid3"]
    obs_perms, act_perms = orc.OracleEnv(kind, n, gs, add_perms=True).twists()
    assert len(obs_perms) == 8 and len(act_perms) == 8
    q = qubit_twist_table(obs_perms, n)
    for k, op in enumerate(obs_perms):
        p = np.argsort(q[k])
        assert op == [int(p[r]) * n + int(p[c]) for r in range(n) for c in range(n)]


# ---- GPU: the decisions re-enacted -----------------------------------------------------------------------------------------------
REENACT = ["C1_perm_grid3", "lf5_line_swap", "clifford3_allgates"]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["fused", "tensor_core"])
@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("name", REENACT)
def test_decisions_reenacted_on_cpu(name, deterministic, backend):
    """Per decision (RolloutSearch.hook): the policy's input bits are the oracle's observation twisted by k = mulhi(philox(seed; g, tick, 5), K)
    with the oracle's obs perms, the frames are those k, and the oracle env driven by cpu_pick(probs[act_perm[k]]) reproduces every rollout's
    return (f32 bits), success and solution, and every target's key and winner."""
    from qiskit_gym_b200.search import RolloutSearch, decode_key
    kind, n, gs, kw = H.config_table()[name]
    pk = dict(kw, add_inverts=False)
    T, R, seed = 3, 40, 123
    states = [r.tolist() for r in H.random_targets(kind, n, gs, T, 5, scramble=2)]
    pol = _policy(kind, n, gs, pk, seed=3, embedding_size=128, common_layers=(64,))
    rs = RolloutSearch(kind, n, gs, pol, R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=T, use_twists=True, **pk)
    obs_perms, act_perms = orc.OracleEnv(kind, n, gs, add_perms=True, **pk).twists()
    K = len(obs_perms)
    assert rs.num_twists == K and K >= 2
    assert np.array_equal(rs.act_table.cpu().numpy(), np.asarray(act_perms, dtype=np.int32))
    act = np.asarray(act_perms, dtype=np.int64)
    rec = []
    rs.hook = lambda probs, bits, twist: rec.append((probs.cpu().numpy().copy(), bits.cpu().numpy().view(np.uint32).copy(), twist.cpu().numpy().copy()))
    res = rs.solve_many(states, deterministic=deterministic, seed=seed)
    assert 1 <= len(rec) <= MAX_DEPTH and all(r.iterations == len(rec) for r in res)
    obs = int(np.prod(rs.env.obs_shape()))
    rets_dev = rs.env.returns().cpu().numpy()
    success_dev = rs.env.status()[2].cpu().numpy()
    sols_dev = rs.env.solutions()
    frames = set()
    for t in range(T):
        keys, sols = [], []
        for j in range(R):
            g = t * R + j
            r = orc.OracleEnv(kind, n, gs, max_depth=MAX_DEPTH, add_perms=False, **pk)
            r.set_state(states[t])
            ret, tick = np.float32(0.0), 0
            for P, bits, tw in rec:
                if r.is_final():
                    break
                k = twist_index(seed, g, tick, K)
                frames.add(k)
                assert tw[g] == k, (t, j, tick)
                want = _pack([obs_perms[k][i] for i in r.observe()], obs)
                assert np.array_equal(bits[g], want), (t, j, tick)
                a = cpu_pick(P[g][act[k]], orc.philox_draw(seed, g, tick, STREAM_SAMPLE), deterministic)
                r.step(a)
                ret = np.float32(ret + np.float32(r.reward()))
                tick += 1
            assert rets_dev[g].view(np.uint32) == ret.view(np.uint32), (t, j)
            assert bool(success_dev[g]) == r.success() and sols_dev[g] == r.solution(), (t, j)
            keys.append(order_key(r.success(), ret, g))
            sols.append(r.solution())
        best = int(np.argmax(keys))
        assert res[t].key == keys[best]
        ok, rid = decode_key(res[t].key)
        assert rid == t * R + best and res[t].success == ok
        assert res[t].actions == (sols[best] if ok else None)
    assert len(frames) == K                                # the rollouts spread over the whole symmetry group


# ---- GPU: one launch == two launches ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,deterministic,inverts", [("C1_perm_grid3", False, False), ("C1_perm_grid3", False, True), ("lf5_line_swap", False, True),
                                                        ("clifford3_allgates", False, False), ("clifford3_allgates", True, True),
                                                        ("clifford16_allgates", False, False)])
def test_persistent_twisted_equals_fused_twisted(name, deterministic, inverts):
    """qg_search_run_twisted takes exactly the decisions of qg_policy_forward_bits + qg_search_step_twisted: keys, solutions, returns (f32
    bits), final states, remaining depths and the last frames.  clifford16 (a dense 1 024-entry observation): the first layer's lists of
    changed entries overflow policy_ent_cap and are processed in row groups."""
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch
    kind, n, gs, kw = H.config_table()[name]
    kw = dict(kw, add_inverts=inverts)
    R = 203
    torch.manual_seed(4)
    probe = orc.OracleEnv(kind, n, gs, add_perms=False, **kw)
    pol = BasicPolicy(probe.obs_shape(), len(gs), embedding_size=64, common_layers=(32,))
    tgt = orc.OracleEnv(kind, n, gs, difficulty=4, add_perms=False, **kw)
    tgt.reset(seed=9, env_id=0)
    state = tgt.raw_state().astype(np.int64).tolist()
    out = {}
    for backend in ("fused", "persistent"):
        rs = RolloutSearch(kind, n, gs, pol, R, max_depth=10, policy_backend=backend, use_cuda_graph=False, use_twists=True, **kw)
        res = rs.solve(state, deterministic=deterministic, seed=5, first_rollout_id=1000)
        out[backend] = (res.key, res.actions, rs.env.returns().cpu().numpy().view(np.uint32).copy(), [rs.env.get_state(b) for b in (0, 7, 8, 100, R - 1)],
                        rs.env.status()[3].cpu().numpy().copy(), res.iterations)
    a, b = out["fused"], out["persistent"]
    assert a[0] == b[0] and a[1] == b[1]
    assert np.array_equal(a[2], b[2])
    assert all(np.array_equal(x, y) for x, y in zip(a[3], b[3]))
    assert np.array_equal(a[4], b[4])
    assert a[5] == b[5]


# ---- GPU: identity table == untwisted ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["persistent", "fused", "tensor_core"])
@pytest.mark.parametrize("name", ["perm", "lf_inv", "clifford"])
def test_identity_table_equals_untwisted(name, backend):
    """A twist table holding only the identity (K = 1) gives the untwisted search's results bit for bit, for solve and solve_many."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config(name)
    states = _targets(name, 6, seed=31)
    pol = _policy(kind, n, gs, kw, seed=8, embedding_size=128, common_layers=(64,))
    mk = lambda twists, tpl: RolloutSearch(kind, n, gs, pol, 37, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=tpl,
                                           use_twists=twists, **kw)
    plain, tw, plain6, tw6 = mk(False, 1), mk(True, 1), mk(False, 6), mk(True, 6)
    for s in (tw, tw6):
        dev = s.env.device
        s.qperm_table = torch.arange(n, dtype=torch.uint8, device=dev).reshape(1, n)
        s.act_table = torch.arange(s.env.num_actions(), dtype=torch.int32, device=dev).reshape(1, -1)
        s.num_twists = 1
    for det in (False, True):
        for seed, first in ((1, 0), (7, 555)):
            a, b = plain.solve(states[0], deterministic=det, seed=seed, first_rollout_id=first), tw.solve(states[0], deterministic=det, seed=seed, first_rollout_id=first)
            assert _same(a, b), (det, seed, first)
            assert np.array_equal(plain.env.returns().cpu().numpy().view(np.uint32), tw.env.returns().cpu().numpy().view(np.uint32))
            assert not tw.twist.any()
        a, b = plain6.solve_many(states, deterministic=det, seed=3), tw6.solve_many(states, deterministic=det, seed=3)
        assert all(_same(x, y) for x, y in zip(a, b)), det


# ---- GPU: the solve_many contract ------------------------------------------------------------------------------------------------
_REFS = {}


def _single(name, backend, R, det, t, state, seed, pol):
    key = (name, backend, R, det, t, seed)
    if key not in _REFS:
        from qiskit_gym_b200.search import RolloutSearch
        rs = _REFS.get(("search", name, backend, R))
        if rs is None:
            kind, n, gs, kw = _config(name)
            rs = RolloutSearch(kind, n, gs, pol, R, max_depth=MAX_DEPTH, policy_backend=backend, use_twists=True, **kw)
            _REFS[("search", name, backend, R)] = rs
        _REFS[key] = rs.solve(state, deterministic=det, seed=seed, first_rollout_id=t * R)
    return _REFS[key]


_POLS = {}


def _pol(name):
    if name not in _POLS:
        kind, n, gs, kw = _config(name)
        _POLS[name] = _policy(kind, n, gs, kw, seed=1, embedding_size=128, common_layers=(64,))
    return _POLS[name]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["persistent", "tensor_core"])
@pytest.mark.parametrize("R", [1, 7, 203])
@pytest.mark.parametrize("name", ["perm", "lf_inv", "clifford"])
def test_solve_many_bit_identical_to_single_target(name, R, backend):
    """Target t of a twisted solve_many equals solve(states[t], first_rollout_id=t*R) of a twisted single-target search: the frames are
    keyed on the global rollout id, not on the launch."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config(name)
    states = _targets(name, 37)
    seed = 5
    for T in (1, 5, 37):
        rs = RolloutSearch(kind, n, gs, _pol(name), R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=T, use_twists=True, **kw)
        for det in (False, True):
            got = rs.solve_many(states[:T], deterministic=det, seed=seed)
            for t in range(T):
                ref = _single(name, backend, R, det, t, states[t], seed, _pol(name))
                assert _same(got[t], ref), (T, det, t, got[t], ref)
                if got[t].success and not kw.get("add_inverts"):
                    assert _replays_to_success(kind, n, gs, kw, states[t], got[t].actions, max_depth=MAX_DEPTH), (T, det, t)
            if T >= 5:
                assert got[1].success and got[1].actions == [] and got[1].rollout_id == R
                assert got[3].actions is None and not got[3].success


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["persistent", "fused", "tensor_core"])
def test_chunking_and_graph_replay(backend):
    """Twisted solve_many does not depend on targets_per_launch; CUDA-graph replay equals launch-by-launch iteration over several (seed,
    first rollout id)."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    R, T = 7, 9
    states = _targets("perm", T, seed=21)
    pol = _pol("perm")
    results = {}
    for tpl in (1, 4, T):
        rs = RolloutSearch(kind, n, gs, pol, R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=tpl, use_twists=True, **kw)
        for det in (False, True):
            results[tpl, det] = rs.solve_many(states, deterministic=det, seed=9)
    for det in (False, True):
        for tpl in (4, T):
            assert all(_same(a, b) for a, b in zip(results[1, det], results[tpl, det])), (tpl, det)
    mk = lambda graph: RolloutSearch(kind, n, gs, pol, 64, max_depth=MAX_DEPTH, policy_backend=backend, use_cuda_graph=graph, use_twists=True, **kw)
    g, e = mk(True), mk(False)
    for seed, first in ((1, 0), (2, 0), (2, 640), (1, 640)):
        a, b = g.solve(states[0], seed=seed, first_rollout_id=first), e.solve(states[0], seed=seed, first_rollout_id=first)
        assert _same(a, b) and np.array_equal(g.env.returns().cpu().numpy(), e.env.returns().cpu().numpy()), (seed, first)
        assert torch.equal(g.twist, e.twist)


# ---- GPU: validity at K = 40 320 ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_validity_c3_all_to_all():
    """C3 (Clifford 8q, all-to-all CX: K = 40 320 qubit symmetries, an 11.6 MB act-perm table), default-shape random policy, one-launch
    twisted search: every returned solution, applied to its target by the oracle, gives the identity."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, _ = H.config_table()["C3_clifford8_full"]
    kw = {"add_inverts": False}
    T, R = 64, 128
    states = [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 1, scramble=1)] + \
             [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 2, scramble=2)]
    pol = _policy(kind, n, gs, kw, seed=1, embedding_size=512, common_layers=(256,))
    rs = RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, use_twists=True, **kw)
    assert rs.num_twists == 40320 and tuple(rs.act_table.shape) == (40320, len(gs))
    res = rs.solve_many(states, seed=17)
    solved = [t for t in range(T) if res[t].success]
    assert len(solved) > 8
    for t in solved:
        assert _replays_to_success(kind, n, gs, kw, states[t], res[t].actions), t
    assert len(set(rs.twist.cpu().tolist())) > 1000


# ---- GPU: public API -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rlsynthesis_use_twists():
    """The 3x3-grid reference checkpoint: synth_many(use_twists=True) equals twisted single-target solves, synth equals its first entry, the
    twisted searches are cached apart from the untwisted ones (whose results do not change), and the tree search refuses twists."""
    import os
    from qiskit_gym_b200.rl import RLSynthesis
    models = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models")
    rls = RLSynthesis.from_config_json(os.path.join(models, "perm_square_3x3.json"), os.path.join(models, "perm_square_3x3.pt"))
    rng = np.random.default_rng(3)
    inputs = [[int(v) for v in rng.permutation(9)] for _ in range(6)]
    R, seed = 32, 4
    plain = rls.synth_many(inputs, num_searches=R, seed=seed)
    got = rls.synth_many(inputs, num_searches=R, seed=seed, use_twists=True)
    single = rls._search(R, use_twists=True)
    assert single.use_twists and single.backend == "persistent" and single.num_twists == 8
    for t, x in enumerate(inputs):
        acts = single.solve(rls.env.get_state(x), seed=seed, first_rollout_id=t * R).actions
        assert got[t] == (None if acts is None else rls.env.build_circuit_from_solution(acts, x)), t
    assert rls.synth(inputs[0], num_searches=R, seed=seed, use_twists=True) == got[0]
    assert sum(g is not None for g in got) >= 4
    assert not rls._search(R).use_twists and rls._search(R) is not single
    assert rls.synth_many(inputs, num_searches=R, seed=seed) == plain
    with pytest.raises(NotImplementedError):
        rls.synth(inputs[0], num_searches=R, num_mcts_searches=4, use_twists=True)
