"""Searches over many targets in one launch (RolloutSearch.solve_many, RLSynthesis.solve_many / synth_many): every target's result is
bit-identical to a single-target search on the same global rollout ids; the grouped load (qg_set_state_grouped) and the per-target winner
reduction (qg_search_best_grouped) against per-env loads and a CPU restatement of the key."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_search import order_key

KINDS = {"perm": "C1_perm_grid3", "lf_inv": "lf5_line_swap", "clifford": "clifford3_allgates", "pauli": "pauli3_line"}
MAX_DEPTH = 8


def _config(name):
    kind, n, gs, kw = H.config_table()[KINDS[name]]
    kw = dict(kw)
    if kind != H.PAULI:
        kw["add_inverts"] = name == "lf_inv"           # LinearFunction with inverts: the search draws coins too
    return kind, n, gs, kw


def _trim(kind, n, rows):
    lens = H.payload_lengths(kind, n, rows)
    return [rows[i, : lens[i]].tolist() for i in range(rows.shape[0])]


def _targets(name, count, seed=11):
    """`count` payloads: [0] shallow, [1] the identity (solved at load), [2] a copy of [0], [3] unreachable within MAX_DEPTH, then shallow."""
    from qiskit_gym_b200.search import identity_payload
    kind, n, gs, kw = _config(name)
    rng = np.random.default_rng(seed)
    if kind == H.PERM:
        swaps = [q for _, q in gs]
        shallow = []
        for _ in range(count):
            p = list(range(n))
            for _ in range(int(rng.integers(1, 4))):
                a, b = swaps[int(rng.integers(len(swaps)))]
                p[a], p[b] = p[b], p[a]
            shallow.append(p)
        far = list(range(n))[::-1]                     # the reversal of the 3x3 grid needs >= 12 swaps
    elif kind == H.PAULI:
        shallow = _trim(kind, n, H.random_targets(kind, n, gs, count, seed, scramble=2, num_rotations=2, vary_rotations=True))
        far = _trim(kind, n, H.random_targets(kind, n, gs, 1, seed + 1, scramble=200, num_rotations=3))[0]
    else:
        shallow = [r.tolist() for r in H.random_targets(kind, n, gs, count, seed, scramble=3)]
        far = H.random_targets(kind, n, gs, 1, seed + 1, scramble=200)[0].tolist()
    out = list(shallow)
    out[1], out[2], out[3] = identity_payload(kind, n), list(out[0]), far
    return out


def _policy(kind, n, gs, kw, seed=0, **shape):
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200.search import BasicPolicy
    probe = BatchedEnv(kind, n, gs, 1, add_perms=False, **kw)
    torch.manual_seed(seed)
    return BasicPolicy(probe.obs_shape(), probe.num_actions(), **(shape or {"embedding_size": 64, "common_layers": (32,)}))


def _loaded_state(kind, n, gs, kw, payload):
    from qiskit_gym_b200 import BatchedEnv
    env = BatchedEnv(kind, n, gs, 1, add_perms=False, **kw)
    env.set_state(payload)
    return env.get_state(0).tolist()


def _replays_to_success(kind, n, gs, kw, state, actions, max_depth=128):
    r = orc.OracleEnv(kind, n, gs, max_depth=max_depth, add_perms=False, **kw)
    r.set_state(state)
    for a in actions:
        r.step(a)
    return r.success()


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_chunk_plan():
    from qiskit_gym_b200.search import chunk_plan
    assert chunk_plan(0, 4, 100) == []
    assert chunk_plan(1, 1, 100) == [(0, 1, 0)]
    plan = chunk_plan(10, 4, 7)
    assert plan == [(0, 4, 0), (4, 4, 28), (8, 2, 56)]
    assert [4 - c for _, c, _ in plan] == [0, 0, 2]              # padding of each chunk
    assert chunk_plan(5, 8, 3) == [(0, 5, 0)]
    assert chunk_plan(3, 1, 5) == [(0, 1, 0), (1, 1, 5), (2, 1, 10)]
    assert chunk_plan(2, 2, (1 << 29) - 1)[-1] == (0, 2, 0)       # 2^30 - 2 rollouts: the last id 2^30 - 3 fits
    for T, R in ((2, 1 << 29), (1, 1 << 30), (1 << 20, 1 << 10), (3, 1 << 29)):
        with pytest.raises(ValueError):
            chunk_plan(T, 1, R)


def test_identity_payload_shapes():
    from qiskit_gym_b200.search import identity_payload
    assert identity_payload(H.PERM, 4) == [0, 1, 2, 3]
    assert identity_payload(H.LF, 2) == [1, 0, 0, 1]
    assert len(identity_payload(H.CLIFF, 3)) == 36 and identity_payload(H.CLIFF, 3)[:7] == [1, 0, 0, 0, 0, 0, 0]
    p = identity_payload(H.PAULI, 2)
    assert p[0] == 0 and len(p) == 17 and np.array_equal(np.array(p[1:]).reshape(4, 4), np.eye(4))


# ---- GPU --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(KINDS))
def test_identity_payload_is_final_at_load(name):
    """What solve_many pads short chunks with: flagged success by k_load, so the slot is final before the first decision."""
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200.search import identity_payload
    kind, n, gs, kw = _config(name)
    env = BatchedEnv(kind, n, gs, 24, add_perms=False, **kw)
    env.set_state_grouped([_targets(name, 4)[3], identity_payload(kind, n)], 12)
    _, done, success, _ = env.status()
    assert not success[:12].any().item() and success[12:].all().item() and done[12:].all().item()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(KINDS))
def test_grouped_load_matches_per_env_load(name):
    from qiskit_gym_b200 import BatchedEnv
    kind, n, gs, kw = _config(name)
    B, group = 50, 11
    payloads = _targets(name, 4, seed=3)
    a = BatchedEnv(kind, n, gs, B, add_perms=False, **kw)
    b = BatchedEnv(kind, n, gs, B, add_perms=False, **kw)
    for e in (a, b):
        e.reset(seed=7)
    a.set_state_grouped(payloads, group)
    b.set_state([p for p in payloads for _ in range(group)])     # per-env payloads for envs 0 .. 43; 44 .. 49 keep their reset state
    for x, y in zip(a.status(), b.status()):
        assert torch.equal(x, y)
    for env in range(B):
        assert np.array_equal(a.get_state(env), b.get_state(env)), env
    c = BatchedEnv(kind, n, gs, B, add_perms=False, **kw)
    c.reset(seed=7)
    for env in range(len(payloads) * group, B):
        assert np.array_equal(a.get_state(env), c.get_state(env))
    for bad_states, bad_group in ((payloads, 0), (payloads, -3), (payloads, 13), (payloads * 13, 1)):
        with pytest.raises(ValueError):
            a.set_state_grouped(bad_states, bad_group)


_REFS = {}


def _single(name, backend, R, deterministic, t, state, seed):
    """Single-target solve of target t (global rollout ids t*R ..), cached over the test's parameters."""
    key = (name, backend, R, deterministic, t, seed)
    if key not in _REFS:
        rs = _REFS.get(("search", name, backend, R))
        if rs is None:
            from qiskit_gym_b200.search import RolloutSearch
            kind, n, gs, kw = _config(name)
            rs = RolloutSearch(kind, n, gs, _policy(kind, n, gs, kw), R, max_depth=MAX_DEPTH, policy_backend=backend, **kw)
            _REFS[("search", name, backend, R)] = rs
        _REFS[key] = rs.solve(state, deterministic=deterministic, seed=seed, first_rollout_id=t * R)
    return _REFS[key]


def _same(a, b):
    return (a.actions, a.key, a.rollout_id, a.success) == (b.actions, b.key, b.rollout_id, b.success)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["persistent", "fused"])
@pytest.mark.parametrize("R", [1, 7, 203])
@pytest.mark.parametrize("name", list(KINDS))
def test_solve_many_bit_identical_to_single_target(name, R, backend):
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config(name)
    states = _targets(name, 37)
    seed = 5
    for T in (1, 5, 37):
        rs = RolloutSearch(kind, n, gs, _policy(kind, n, gs, kw), R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=T, **kw)
        if T > 1:
            with pytest.raises(ValueError):
                rs.solve(states[0])
        for det in (False, True):
            got = rs.solve_many(states[:T], deterministic=det, seed=seed)
            assert len(got) == T
            for t in range(T):
                ref = _single(name, backend, R, det, t, states[t], seed)
                assert _same(got[t], ref), (T, det, t, got[t], ref)
                assert got[t].rollouts == R
            if T >= 5:
                assert got[1].success and got[1].actions == [] and got[1].rollout_id == R          # solved at load: the lowest id wins
                assert got[3].actions is None and not got[3].success                               # unreachable
    with pytest.raises(ValueError):
        RolloutSearch(kind, n, gs, _policy(kind, n, gs, kw), R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=0, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["persistent", "fused"])
@pytest.mark.parametrize("name", ["perm", "pauli"])
def test_chunking_does_not_matter(name, backend):
    from qiskit_gym_b200.search import RolloutSearch, identity_payload
    kind, n, gs, kw = _config(name)
    R, T = 7, 8
    states = _targets(name, T, seed=21)
    pol = _policy(kind, n, gs, kw, seed=4)
    results = {}
    for tpl in (1, 3, T):
        rs = RolloutSearch(kind, n, gs, pol, R, max_depth=MAX_DEPTH, policy_backend=backend, targets_per_launch=tpl, **kw)
        results[tpl] = rs.solve_many(states, seed=9)
        if tpl == 3:
            # the last chunk held targets 6, 7 and one padded slot: loaded as solved, never stepped
            _, done, success, depth = rs.env.status()
            assert success[2 * R: 3 * R].all().item() and done[2 * R: 3 * R].all().item()
            assert (depth[2 * R: 3 * R] == MAX_DEPTH).all().item()
            assert (rs.env.returns()[2 * R: 3 * R] == 0).all().item()
            assert rs.env.solutions(2 * R, R) == [[]] * R
            assert rs.env.get_state(2 * R).tolist() == _loaded_state(kind, n, gs, kw, identity_payload(kind, n))
    for tpl in (3, T):
        assert all(_same(a, b) for a, b in zip(results[1], results[tpl])), tpl
    assert any(r.success for r in results[1]) and not results[1][3].success


@pytest.mark.gpu
@pytest.mark.parametrize("deterministic", [False, True])
def test_grouped_winner_against_cpu_restatement(deterministic):
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    R, T = 7, 9
    states = _targets("perm", T, seed=31)
    rs = RolloutSearch(kind, n, gs, _policy(kind, n, gs, kw, seed=2), R, max_depth=MAX_DEPTH, targets_per_launch=T, **kw)
    res = rs.solve_many(states, deterministic=deterministic, seed=3)
    env = rs.env
    rets = env.returns().cpu().numpy()
    _, _, success, _ = env.status()
    success = success.cpu().numpy()
    sols = env.solutions()
    keys = [order_key(bool(success[e]), rets[e], e) for e in range(T * R)]
    dkeys, dlens, dacts = (x.cpu().numpy() for x in env.search_best_grouped(R, T))
    saw_fail = saw_tie = False
    for g in range(T):
        grp = keys[g * R: (g + 1) * R]
        best = max(grp)
        w = g * R + grp.index(best)
        assert int(dkeys[g]) == best == res[g].key and res[g].rollout_id == w
        ties = [e for e in range(g * R, (g + 1) * R) if bool(success[e]) == bool(success[w]) and rets[e] == rets[w]]
        assert w == min(ties)
        saw_tie |= len(ties) > 1
        if success[w]:
            assert dlens[g] == len(sols[w]) and dacts[g, : dlens[g]].tolist() == sols[w] == res[g].actions
        else:
            saw_fail = True
            assert dlens[g] == 0 and res[g].actions is None
    assert saw_fail                                              # the unreachable target
    if deterministic:
        assert saw_tie                                           # identical rollouts: the lowest id wins
        assert all(res[g].rollout_id == g * R for g in range(T))
    # cap too small: -(length) and nothing written
    marker = torch.full((T * (3 + 1),), -7, dtype=torch.int32, device=env.device)
    _, lens1, acts1 = env.search_best_grouped(R, T, cap=1, out=marker)
    lens1, acts1 = lens1.cpu().numpy(), acts1.cpu().numpy()
    for g in range(T):
        n_ = len(res[g].actions) if res[g].actions is not None else 0
        if res[g].actions is None:
            assert lens1[g] == 0 and acts1[g, 0] == -7
        elif n_ > 1:
            assert lens1[g] == -n_ and acts1[g, 0] == -7
        else:
            assert lens1[g] == n_
    if not deterministic:
        assert any(lens1 < 0)
    # fewer groups than the batch holds, and groups that straddle targets
    k2, l2, a2 = env.search_best_grouped(3, 10, cap=64)
    for g in range(10):
        grp = keys[g * 3: (g + 1) * 3]
        assert int(k2[g].item()) == max(grp)
    for bad in ((0, 1), (R, T + 1), (T * R + 1, 1), (-1, 1)):
        with pytest.raises(ValueError):
            env.search_best_grouped(*bad)
    with pytest.raises(ValueError):
        env.search_best_grouped(R, T, cap=0)


@pytest.mark.gpu
def test_collector_scale_one_launch():
    """C3 (Clifford 8q, all-to-all CX): 512 targets x 128 rollouts in one launch with the default-shape random-weight policy."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, _ = H.config_table()["C3_clifford8_full"]
    kw = {"add_inverts": False}
    T, R = 512, 128
    rng = np.random.default_rng(0)
    states = [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 1, scramble=1)] + \
             [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 2, scramble=2)]
    order = rng.permutation(T)
    states = [states[i] for i in order]
    pol = _policy(kind, n, gs, kw, seed=1, embedding_size=512, common_layers=(256,))
    rs = RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, **kw)
    assert rs.env.batch == 65536
    res = rs.solve_many(states, seed=17)
    solved = [t for t in range(T) if res[t].success]
    assert len(solved) > 50
    for t in solved:
        assert _replays_to_success(kind, n, gs, kw, states[t], res[t].actions)
    single = RolloutSearch(kind, n, gs, pol, R, **kw)
    for t in list(rng.choice(T, 8, replace=False)):
        assert _same(res[t], single.solve(states[t], seed=17, first_rollout_id=int(t) * R)), t


@pytest.mark.gpu
def test_torch_backend_valid_results():
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    states = _targets("perm", 7, seed=41)
    rs = RolloutSearch(kind, n, gs, _policy(kind, n, gs, kw), 256, max_depth=MAX_DEPTH, policy_backend="torch", targets_per_launch=3, **kw)
    res = rs.solve_many(states, seed=2)
    assert len(res) == 7 and res[3].actions is None and res[1].actions == []
    assert sum(r.success for t, r in enumerate(res) if t != 1) >= 1            # (besides the target that is solved at load)
    for s, r in zip(states, res):
        assert (r.actions is None) == (not r.success)
        if r.success:
            assert _replays_to_success(kind, n, gs, kw, s, r.actions, max_depth=MAX_DEPTH)


@pytest.mark.gpu
def test_rlsynthesis_synth_many_clifford_with_phase():
    import os
    from qiskit_gym_b200 import wire
    from qiskit_gym_b200.rl import RLSynthesis
    models = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models")
    rls = RLSynthesis.from_config_json(os.path.join(models, "clifford_3q_custom.json"), os.path.join(models, "clifford_3q_custom.pt"))
    n = rls.env_config["num_qubits"]
    gs = [(g, tuple(q)) for g, q in rls.env_config["gateset"]]
    rng = np.random.default_rng(8)
    inputs = []
    for i in range(6):
        tg = [gs[int(rng.integers(len(gs)))] for _ in range(6)]
        if i % 2 == 0:                                   # Pauli gates: a tableau with a phase column
            tg.insert(int(rng.integers(len(tg))), (("x", "y", "z")[i % 3], (int(rng.integers(n)),)))
            inputs.append(tg)
        else:
            inputs.append(wire.StabilizerTableau.from_gates(tg, n).to_array()[:, : 2 * n])
    R, seed = 32, 4
    got = rls.synth_many(inputs, num_searches=R, seed=seed)
    assert got[0] == rls.synth(inputs[0], num_searches=R, seed=seed)
    single = rls._search(R)
    for t, x in enumerate(inputs):
        acts = single.solve(rls.env.get_state(x), seed=seed, first_rollout_id=t * R).actions
        assert got[t] == (None if acts is None else rls.env.build_circuit_from_solution(acts, x)), t
    assert sum(g is not None for g in got) >= 4
    # the same with several targets per launch bounded by max_rollouts
    assert rls.synth_many(inputs, num_searches=R, seed=seed, max_rollouts=2 * R) == got
    with pytest.raises(NotImplementedError):
        rls.synth_many(inputs, num_searches=R, num_mcts_searches=4)
    with pytest.raises(ValueError):
        rls.synth_many(inputs[:2], num_searches=1 << 29)
    with pytest.raises(ValueError):
        rls.solve_many([rls.env.get_state(inputs[0])], num_searches=1 << 30)


@pytest.mark.gpu
def test_rlsynthesis_synth_many_pauli_network_rotation_sets():
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    tri = [(0, 1), (1, 0), (1, 2), (2, 1)]
    spec = SynthSpec.from_coupling_map("PauliNetworkEnv", tri, basis_gates=("H", "S", "SX", "CX"), max_depth=16)
    rls = RLSynthesis(spec, {}, {"embedding_size": 64, "common_layers": [32]})
    inputs = [([], ["ZZI"]), ([("h", (0,))], []), ([], ["XXI", "IZZ"]), ([("cx", (0, 1))], ["ZIZ"]), ([], []), ([("s", (2,))], ["YII", "IXX", "ZZZ"])]
    R, seed = 64, 6
    got = rls.synth_many(inputs, num_searches=R, seed=seed)
    assert got[0] == rls.synth(inputs[0], num_searches=R, seed=seed)
    single = rls._search(R)
    for t, x in enumerate(inputs):
        acts = single.solve(spec.get_state(x), seed=seed, first_rollout_id=t * R).actions
        spec.get_state(x)
        assert got[t] == (None if acts is None else spec.build_circuit_from_solution(acts, x)), t
    assert got[4] == [] and sum(g is not None for g in got) >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["fused", "torch"])
def test_graph_replay_honours_seed_and_first_rollout_id(backend):
    """The captured iteration's launches carry the seed and first rollout id of their capture: a search with other ones re-captures,
    so graph replay and launch-by-launch runs agree for every (seed, first_rollout_id)."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    state = _targets("perm", 5, seed=51)[0]
    pol = _policy(kind, n, gs, kw, seed=6)
    g = RolloutSearch(kind, n, gs, pol, 64, max_depth=MAX_DEPTH, policy_backend=backend, **kw)
    e = RolloutSearch(kind, n, gs, pol, 64, max_depth=MAX_DEPTH, policy_backend=backend, use_cuda_graph=False, **kw)
    for seed, first in ((1, 0), (2, 0), (2, 640), (1, 640)):
        a, b = g.solve(state, seed=seed, first_rollout_id=first), e.solve(state, seed=seed, first_rollout_id=first)
        assert _same(a, b) and np.array_equal(g.env.returns().cpu().numpy(), e.env.returns().cpu().numpy()), (seed, first)
