"""The "tensor_core" search backend (RolloutSearch(policy_backend="tensor_core"), RLSynthesis.solve_many / synth_many(matmul_precision=
"tensor_core")).  Its many-target contract rests on one property of the tensor-core policy, tested first: a row's probabilities are
bit-identical whatever the batch size, the handle's capacity, the row's position and the rows around it.  Then: solve_many against
single-target solves on the same backend, the step's decisions re-enacted on the CPU from the probabilities it consumed (and those
probabilities against the float64 module), validity at collector scale, and the public API."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_policy_tc_envelope import Refs, make_policy
from tests.test_search import STREAM_SAMPLE, cpu_pick, order_key
from tests.test_search_many import KINDS, MAX_DEPTH, _config, _policy, _replays_to_success, _same, _targets

# network per env kind: a fused three-layer shape (embedding a multiple of 128) and the per-layer path (64-wide embedding)
SHAPES = {"perm": {"embedding_size": 128, "common_layers": (64,)}, "clifford": {"embedding_size": 128, "common_layers": (64,)},
          "lf_inv": {}, "pauli": {}}
FUSED = {"perm": True, "clifford": True, "lf_inv": False, "pauli": False}


def _dev():
    return torch.device("cuda", 0)


def _random_bits(rng, B, obs):
    """Packed observations int32 [B, ceil(obs / 32)] with random entries and the bits past obs clear (as observe_bits leaves them)."""
    words = (obs + 31) // 32
    w = rng.integers(0, 1 << 32, size=(B, words), dtype=np.uint64).astype(np.uint32)
    if obs % 32:
        w[:, -1] &= np.uint32((1 << (obs % 32)) - 1)
    return torch.from_numpy(w.view(np.int32)).to(_dev())


def _unpack(bits, obs):
    u = np.ascontiguousarray(bits.cpu().numpy()).view(np.uint32)
    n = u.shape[0]
    return torch.from_numpy(np.unpackbits(u.view(np.uint8).reshape(n, -1), axis=1, bitorder="little")[:, :obs].astype(np.float32))


_POLICIES = {}


def _tc_policy(name):
    if name not in _POLICIES:
        kind, n, gs, kw = _config(name)
        _POLICIES[name] = _policy(kind, n, gs, kw, seed=1, **SHAPES[name])
    return _POLICIES[name]


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_refusals_before_any_device_work():
    """matmul_precision is checked, and the tensor-core search's limits are refused up front, without a device."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.search import check_tensor_core_search
    from qiskit_gym_b200.specs import SynthSpec
    m = 17                                            # 136 SWAP actions: more than the tensor-core head's 127
    spec = SynthSpec.from_coupling_map("PermutationEnv", [(i, j) for i in range(m) for j in range(i + 1, m)], max_depth=8)
    assert spec.num_actions() == 136
    rls = RLSynthesis(spec, {}, {"embedding_size": 64, "common_layers": [32]})
    with pytest.raises(NotImplementedError):
        rls.synth_many([list(range(m))], num_searches=4, matmul_precision="tensor_core")
    with pytest.raises(ValueError):
        rls.synth_many([list(range(m))], num_searches=4, matmul_precision="bf16")
    with pytest.raises(NotImplementedError):
        rls.synth_many([list(range(m))], num_searches=4, num_mcts_searches=2, matmul_precision="tensor_core")
    with pytest.raises(NotImplementedError):
        check_tensor_core_search(H.PERM, 65, 64)      # no packed observations past 64 qubits
    with pytest.raises(NotImplementedError):
        check_tensor_core_search(H.CLIFF, 8, 128)


# ---- GPU: the premise ----------------------------------------------------------------------------------------------------------
ROW_SHAPES = {   # name: (obs, A, E, common, fused)
    "C3": (256, 72, 512, (256,), True),
    "fused_small": (81, 12, 128, (64,), True),
    "per_layer": (81, 12, 300, (256,), False),
    "per_layer_small": (36, 8, 64, (32,), False),
}
ROW_BATCHES = (1, 7, 127, 128, 129, 1184, 65536)
MAX_BATCH = 65536 + 77


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ROW_SHAPES))
def test_rows_bit_identical_across_batches(name):
    """64 fixed observation rows, placed at random positions of batches of every size solve_many produces (one row, a partial tile, one
    CTA wave of the FFMA search, 65 536, the handle's capacity) with random rows around them, through a handle of capacity MAX_BATCH
    and through one of capacity B: every row's probabilities are the bits it has alone in a 64-row batch, in both kernel modes."""
    from qiskit_gym_b200.policy import TensorCorePolicy
    obs, A, E, common, fused = ROW_SHAPES[name]
    dev = _dev()
    rng = np.random.Generator(np.random.PCG64(obs * 7 + A))
    pol = make_policy(obs, A, E, common, seed=5).to(dev)
    big = TensorCorePolicy(pol, max_batch=MAX_BATCH, device=dev, with_value=False)
    assert big.set_per_layer(False) == fused
    K = 64
    fixed = _random_bits(rng, K, obs)
    for per_layer in ([False, True] if fused else [True]):
        big.set_per_layer(per_layer)
        ref = torch.empty((K, A), dtype=torch.float32, device=dev)
        big.forward_bits(fixed, probs=ref)
        Refs(pol, _unpack(fixed, obs).to(dev), with_value=False).check(K, probs=ref, tag=(name, per_layer))
        ref = ref.view(torch.int32)
        for i, B in enumerate(ROW_BATCHES + (MAX_BATCH,)):
            k = min(K, B)
            which = torch.from_numpy((np.arange(k) + 13 * i) % K).to(dev)
            pos = torch.from_numpy(rng.choice(B, size=k, replace=False)).to(dev)
            bits = _random_bits(rng, B, obs)
            bits[pos] = fixed[which]
            handles = [big] + ([TensorCorePolicy(pol, max_batch=B, device=dev, with_value=False)] if B != MAX_BATCH else [])
            for h in handles:
                h.set_per_layer(per_layer)
                out = torch.full(((B + 64) * A,), -7.25, device=dev)
                h.forward_bits(bits, probs=out[: B * A].view(B, A))
                assert bool((out[B * A:] == -7.25).all()), ("wrote past the batch", B)
                got = out[: B * A].view(B, A).view(torch.int32)[pos]
                assert torch.equal(got, ref[which]), (name, per_layer, B, h.max_batch)


# ---- GPU: the contract ---------------------------------------------------------------------------------------------------------
_REFS = {}


def _single(name, R, deterministic, t, state, seed):
    """Single-target "tensor_core" solve of target t (global rollout ids t*R ..), cached over the test's parameters."""
    key = (name, R, deterministic, t, seed)
    if key not in _REFS:
        rs = _REFS.get(("search", name, R))
        if rs is None:
            from qiskit_gym_b200.search import RolloutSearch
            kind, n, gs, kw = _config(name)
            rs = RolloutSearch(kind, n, gs, _tc_policy(name), R, max_depth=MAX_DEPTH, policy_backend="tensor_core", **kw)
            _REFS[("search", name, R)] = rs
        _REFS[key] = rs.solve(state, deterministic=deterministic, seed=seed, first_rollout_id=t * R)
    return _REFS[key]


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 7, 203])
@pytest.mark.parametrize("name", list(KINDS))
def test_solve_many_bit_identical_to_single_target(name, R):
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config(name)
    states = _targets(name, 37)
    seed = 5
    for T in (1, 5, 37):
        rs = RolloutSearch(kind, n, gs, _tc_policy(name), R, max_depth=MAX_DEPTH, policy_backend="tensor_core", targets_per_launch=T, **kw)
        assert rs.handle.max_batch == T * R and rs.handle.set_per_layer(False) == FUSED[name]
        for det in (False, True):
            got = rs.solve_many(states[:T], deterministic=det, seed=seed)
            assert len(got) == T
            for t in range(T):
                ref = _single(name, R, det, t, states[t], seed)
                assert _same(got[t], ref), (T, det, t, got[t], ref)
                assert got[t].rollouts == R
                if got[t].success and not kw.get("add_inverts"):       # (the oracle replays no coin draws)
                    assert _replays_to_success(kind, n, gs, kw, states[t], got[t].actions, max_depth=MAX_DEPTH), (T, det, t)
            if T >= 5:
                assert got[1].success and got[1].actions == [] and got[1].rollout_id == R          # solved at load: the lowest id wins
                assert got[3].actions is None and not got[3].success                               # unreachable


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["perm", "pauli"])
def test_chunking_does_not_matter(name):
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config(name)
    R, T = 7, 9
    states = _targets(name, T, seed=21)
    results = {}
    for tpl in (1, 4, T):
        rs = RolloutSearch(kind, n, gs, _tc_policy(name), R, max_depth=MAX_DEPTH, policy_backend="tensor_core", targets_per_launch=tpl, **kw)
        for det in (False, True):
            results[tpl, det] = rs.solve_many(states, deterministic=det, seed=9)
    for det in (False, True):
        for tpl in (4, T):
            assert all(_same(a, b) for a, b in zip(results[1, det], results[tpl, det])), (tpl, det)
    assert any(r.success for r in results[1, False]) and not results[1, False][3].success


@pytest.mark.gpu
def test_graph_replay_and_weight_refresh():
    """Graph replay equals launch-by-launch runs for solve and solve_many over several (seed, first rollout id); an in-place weight
    update is copied into the handle before the next search without capturing again, and then equals a search built on the new weights."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    states = _targets("perm", 6, seed=51)
    pol = _policy(kind, n, gs, kw, seed=6, embedding_size=128, common_layers=(64,))
    mk = lambda graph, tpl: RolloutSearch(kind, n, gs, pol, 64, max_depth=MAX_DEPTH, policy_backend="tensor_core", use_cuda_graph=graph,
                                          targets_per_launch=tpl, **kw)
    g1, e1, g3, e3 = mk(True, 1), mk(False, 1), mk(True, 3), mk(False, 3)
    for seed, first in ((1, 0), (2, 0), (2, 640), (1, 640)):
        a, b = g1.solve(states[0], seed=seed, first_rollout_id=first), e1.solve(states[0], seed=seed, first_rollout_id=first)
        assert _same(a, b) and np.array_equal(g1.env.returns().cpu().numpy(), e1.env.returns().cpu().numpy()), (seed, first)
    for det in (False, True):
        a, b = g3.solve_many(states, deterministic=det, seed=4), e3.solve_many(states, deterministic=det, seed=4)
        assert all(_same(x, y) for x, y in zip(a, b)), det
    g1.solve(states[0], seed=1)
    before = g1.probs.clone()
    graph = g1._graphs[False][0]
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(-1.5)
    after = g1.solve(states[0], seed=1)
    assert g1._graphs[False][0] is graph              # the captured graph replayed the refreshed weights
    assert not torch.equal(g1.probs, before)
    fresh = mk(False, 1)
    assert _same(after, fresh.solve(states[0], seed=1))
    assert torch.equal(g1.probs, fresh.probs)


# ---- GPU: the decisions re-enacted -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,deterministic", [("C1_perm_grid3", False), ("C1_perm_grid3", True), ("clifford3_allgates", False),
                                                ("pauli3_line", False), ("lf5_line_swap", False)])
def test_decisions_reenacted_on_cpu(name, deterministic):
    """Every decision's probability rows, as the step consumed them (RolloutSearch.hook), drive oracle envs through cpu_pick with the
    same Philox draws: every rollout's actions, f32 return and success, and every target's key and solution, bit for bit.  The rows
    themselves are within TensorCorePolicy's bound of the float64 module."""
    from qiskit_gym_b200.search import RolloutSearch, decode_key
    kind, n, gs, kw = H.config_table()[name]
    pk = dict(kw)
    if kind != H.PAULI:
        pk["add_inverts"] = False
    T, R, seed = 5, 48, 77
    rng = np.random.Generator(np.random.PCG64(len(name)))
    if kind == H.PAULI:
        rows = H.random_targets(kind, n, gs, T, 3, scramble=2, num_rotations=2)
        lens = H.payload_lengths(kind, n, rows)
        states = [rows[i, : lens[i]].tolist() for i in range(T)]
    else:
        states = [r.tolist() for r in H.random_targets(kind, n, gs, T, 3, scramble=2)]
    pol = _policy(kind, n, gs, pk, seed=2, embedding_size=128, common_layers=(64,))
    rs = RolloutSearch(kind, n, gs, pol, R, max_depth=MAX_DEPTH, policy_backend="tensor_core", targets_per_launch=T, **pk)
    rec = []
    rs.hook = lambda probs, bits: rec.append((probs.clone(), bits.clone()))
    res = rs.solve_many(states, deterministic=deterministic, seed=seed)
    assert 1 <= len(rec) <= MAX_DEPTH and all(r.iterations == len(rec) for r in res)
    probs = [p.cpu().numpy() for p, _ in rec]
    rets_dev = rs.env.returns().cpu().numpy()
    _, _, success_dev, _ = rs.env.status()
    success_dev = success_dev.cpu().numpy()
    sols_dev = rs.env.solutions()
    for t in range(T):
        keys, sols = [], []
        for j in range(R):
            g = t * R + j
            r = orc.OracleEnv(kind, n, gs, max_depth=MAX_DEPTH, add_perms=False, **pk)
            r.set_state(states[t])
            ret, tick = np.float32(0.0), 0
            for P in probs:
                if r.is_final():
                    break
                a = cpu_pick(P[g], orc.philox_draw(seed, g, tick, STREAM_SAMPLE), deterministic)
                r.step(a)
                ret = np.float32(ret + np.float32(r.reward()))
                tick += 1
            assert r.is_final() or len(probs) == MAX_DEPTH
            assert rets_dev[g].view(np.uint32) == ret.view(np.uint32), (t, j)
            assert bool(success_dev[g]) == r.success() and sols_dev[g] == r.solution(), (t, j)
            keys.append(order_key(r.success(), ret, g))
            sols.append(r.solution())
        best = int(np.argmax(keys))
        assert res[t].key == keys[best] == max(keys)
        ok, rid = decode_key(res[t].key)
        assert rid == t * R + best and res[t].success == ok
        assert res[t].actions == (sols[best] if ok else None)
    obs = int(np.prod(rs.env.obs_shape()))
    for d, (P, bits) in enumerate(rec):
        sample = torch.from_numpy(np.unique(np.concatenate([[0, T * R - 1], rng.choice(T * R, 64, replace=False)]))).to(rs.env.device)
        Refs(pol, _unpack(bits[sample], obs).to(rs.env.device), with_value=False).check(len(sample), probs=P[sample].contiguous(), tag=d)


# ---- GPU: validity at scale ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_collector_scale_validity():
    """C3 (Clifford 8q, all-to-all CX): 512 targets x 128 rollouts in one tensor-core launch with the default-shape random-weight policy
    (the fused three-layer kernel): every solution replays to its target; sampled targets equal single-target tensor-core solves."""
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, _ = H.config_table()["C3_clifford8_full"]
    kw = {"add_inverts": False}
    T, R = 512, 128
    rng = np.random.default_rng(0)
    states = [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 1, scramble=1)] + \
             [r.tolist() for r in H.random_targets(kind, n, gs, T // 2, 2, scramble=2)]
    states = [states[i] for i in rng.permutation(T)]
    pol = _policy(kind, n, gs, kw, seed=1, embedding_size=512, common_layers=(256,))
    rs = RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, policy_backend="tensor_core", **kw)
    assert rs.env.batch == 65536 and rs.handle.set_per_layer(False)
    res = rs.solve_many(states, seed=17)
    solved = [t for t in range(T) if res[t].success]
    assert len(solved) > 50
    for t in solved:
        assert _replays_to_success(kind, n, gs, kw, states[t], res[t].actions)
    single = RolloutSearch(kind, n, gs, pol, R, policy_backend="tensor_core", **kw)
    for t in list(rng.choice(T, 8, replace=False)):
        assert _same(res[t], single.solve(states[t], seed=17, first_rollout_id=int(t) * R)), t


# ---- GPU: public API -----------------------------------------------------------------------------------------------------------
def _clifford_inputs(rls, count, seed):
    from qiskit_gym_b200 import wire
    n = rls.env_config["num_qubits"]
    gs = [(g, tuple(q)) for g, q in rls.env_config["gateset"]]
    rng = np.random.default_rng(seed)
    inputs = []
    for i in range(count):
        tg = [gs[int(rng.integers(len(gs)))] for _ in range(6)]
        if i % 2 == 0:                                   # Pauli gates: a tableau with a phase column
            tg.insert(int(rng.integers(len(tg))), (("x", "y", "z")[i % 3], (int(rng.integers(n)),)))
            inputs.append(tg)
        else:
            inputs.append(wire.StabilizerTableau.from_gates(tg, n).to_array()[:, : 2 * n])
    return inputs


@pytest.mark.gpu
def test_rlsynthesis_synth_many_tensor_core_clifford():
    import os
    from qiskit_gym_b200.rl import RLSynthesis
    models = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models")
    rls = RLSynthesis.from_config_json(os.path.join(models, "clifford_3q_custom.json"), os.path.join(models, "clifford_3q_custom.pt"))
    inputs = _clifford_inputs(rls, 6, 8)
    R, seed = 32, 4
    got = rls.synth_many(inputs, num_searches=R, seed=seed, matmul_precision="tensor_core")
    tc_single = rls._search(R, matmul_precision="tensor_core")
    assert tc_single.backend == "tensor_core"
    for t, x in enumerate(inputs):
        acts = tc_single.solve(rls.env.get_state(x), seed=seed, first_rollout_id=t * R).actions
        assert got[t] == (None if acts is None else rls.env.build_circuit_from_solution(acts, x)), t
    assert sum(g is not None for g in got) >= 4
    assert rls.synth_many(inputs[:1], num_searches=R, seed=seed, matmul_precision="tensor_core")[0] == got[0]
    assert rls.synth_many(inputs, num_searches=R, seed=seed, max_rollouts=2 * R, matmul_precision="tensor_core") == got
    # the default stays the f32 search, cached apart: synth_many equals a loop of synth's search
    f32 = rls.synth_many(inputs, num_searches=R, seed=seed)
    single = rls._search(R)
    assert single.backend != "tensor_core" and rls._search(R, 6).backend != "tensor_core"
    assert f32[0] == rls.synth(inputs[0], num_searches=R, seed=seed)
    for t, x in enumerate(inputs):
        acts = single.solve(rls.env.get_state(x), seed=seed, first_rollout_id=t * R).actions
        assert f32[t] == (None if acts is None else rls.env.build_circuit_from_solution(acts, x)), t
    assert rls._search(R, 6, "tensor_core") is rls._searches[("tensor_core", ("many", R))]


@pytest.mark.gpu
def test_rlsynthesis_synth_many_tensor_core_pauli_network():
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    tri = [(0, 1), (1, 0), (1, 2), (2, 1)]
    spec = SynthSpec.from_coupling_map("PauliNetworkEnv", tri, basis_gates=("H", "S", "SX", "CX"), max_depth=16)
    rls = RLSynthesis(spec, {}, {"embedding_size": 64, "common_layers": [32]})
    inputs = [([], ["ZZI"]), ([("h", (0,))], []), ([], ["XXI", "IZZ"]), ([("cx", (0, 1))], ["ZIZ"]), ([], []), ([("s", (2,))], ["YII", "IXX", "ZZZ"])]
    R, seed = 64, 6
    got = rls.synth_many(inputs, num_searches=R, seed=seed, matmul_precision="tensor_core")
    single = rls._search(R, matmul_precision="tensor_core")
    for t, x in enumerate(inputs):
        acts = single.solve(spec.get_state(x), seed=seed, first_rollout_id=t * R).actions
        spec.get_state(x)
        assert got[t] == (None if acts is None else spec.build_circuit_from_solution(acts, x)), t
    assert got[4] == [] and sum(g is not None for g in got) >= 3
    with pytest.raises(NotImplementedError):
        rls.synth_many(inputs, num_searches=R, num_mcts_searches=4, matmul_precision="tensor_core")
