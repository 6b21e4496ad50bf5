"""Every consumer of a device policy handle (policy.FusedPolicy / TensorCorePolicy) runs the weights its module holds now: after an in-place
update of the module, and after another module of the same shape is put in its place, whose weights_version can be the old module's."""
import copy

import numpy as np
import pytest
import torch

from tests.test_collector_packed import make_env, rollout_fields
from tests.test_search_many import MAX_DEPTH, _config, _policy, _same, _targets


def _returns(rs):
    return rs.env.returns().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["fused", "persistent"])
def test_search_picks_up_an_in_place_update(backend):
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    state = _targets("perm", 4, seed=3)[0]
    pol = _policy(kind, n, gs, kw, seed=4)

    def mk():
        return RolloutSearch(kind, n, gs, pol, 256, max_depth=MAX_DEPTH, policy_backend=backend, **kw)

    rs = mk()
    rs.solve(state, seed=2)
    before = _returns(rs)
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(-1.5)
    after = rs.solve(state, seed=2)
    fresh = mk()
    want = fresh.solve(state, seed=2)
    assert not np.array_equal(_returns(fresh), before)          # (the update changes the search)
    assert _same(after, want) and np.array_equal(_returns(rs), _returns(fresh))


@pytest.mark.gpu
def test_tensor_core_search_picks_up_another_module():
    from qiskit_gym_b200.policy import weights_version
    from qiskit_gym_b200.search import RolloutSearch
    kind, n, gs, kw = _config("perm")
    states = _targets("perm", 4, seed=5)
    shape = {"embedding_size": 128, "common_layers": (64,)}
    dev = torch.device("cuda", 0)
    pol, other = _policy(kind, n, gs, kw, seed=1, **shape).to(dev), _policy(kind, n, gs, kw, seed=2, **shape).to(dev)
    assert weights_version(other) == weights_version(pol)      # the version alone cannot tell the two apart

    def mk(p, tpl=1):
        return RolloutSearch(kind, n, gs, p, 64, max_depth=MAX_DEPTH, policy_backend="tensor_core", targets_per_launch=tpl, **kw)

    rs, rs_many = mk(pol), mk(pol, 4)
    rs.solve(states[0], seed=1)
    before = _returns(rs)
    rs_many.solve_many(states, seed=1)
    rs.policy, rs_many.policy = other, other
    after, after_many = rs.solve(states[0], seed=1), rs_many.solve_many(states, seed=1)
    fresh, fresh_many = mk(other), mk(other, 4)
    want, want_many = fresh.solve(states[0], seed=1), fresh_many.solve_many(states, seed=1)
    assert not np.array_equal(_returns(fresh), before)
    assert _same(after, want) and np.array_equal(_returns(rs), _returns(fresh)) and torch.equal(rs.probs, fresh.probs)
    assert all(_same(a, b) for a, b in zip(after_many, want_many))


@pytest.mark.gpu
def test_packed_collector_picks_up_another_module():
    """The collector's policy replaced by a same-shape module of another seed: the next rollout equals that of a collector whose module
    received the new weights in place (its captured graph kept)."""
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.policy import weights_version
    from qiskit_gym_b200.search import BasicPolicy
    B, T = 1500, 5
    envs = [make_env("C1_perm_grid3", B, difficulty=3, max_depth=6, depth_slope=2)[0] for _ in range(2)]
    dev = envs[0].device
    torch.manual_seed(4)
    pol = BasicPolicy(envs[0].obs_shape(), envs[0].num_actions(), embedding_size=128, common_layers=(64,)).to(dev)
    torch.manual_seed(5)
    other = BasicPolicy(envs[0].obs_shape(), envs[0].num_actions(), embedding_size=128, common_layers=(64,)).to(dev)
    assert weights_version(other) == weights_version(pol)
    ref_pol = copy.deepcopy(pol)
    col = RolloutCollector(envs[0], pol, seed=5)
    ref = RolloutCollector(envs[1], ref_pol, seed=5)
    for _ in range(2):
        col.collect_packed(T)
        ref.collect_packed(T)
    col.policy = other
    with torch.no_grad():
        for a, b in zip(ref_pol.parameters(), other.parameters()):
            a.copy_(b)
    got, want = rollout_fields(col.collect_packed(T)), rollout_fields(ref.collect_packed(T))
    for x, y in zip(got, want):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_rlsynthesis_cached_search_picks_up_load_state_dict():
    """load_state_dict after a synth: the next synth runs the new weights on the same cached search (no new engine)."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    env = SynthSpec.from_coupling_map("PermutationEnv", [(i, i + 1) for i in range(5)], difficulty=1, depth_slope=2, max_depth=24)
    mc = {"embedding_size": 64, "common_layers": [32]}
    torch.manual_seed(0)
    rls = RLSynthesis(env, {}, mc, device=0)
    torch.manual_seed(1)
    other = RLSynthesis(env, {}, mc, device=0).policy.state_dict()
    targets = [list(np.random.Generator(np.random.PCG64(s)).permutation(6)) for s in range(6)]
    R = 200
    rls.synth(targets[0], num_searches=R, seed=3)
    rs = rls._searches[R]
    before = _returns(rs)
    rls.policy.load_state_dict(other)
    got = [rls.synth(t, num_searches=R, seed=3) for t in targets]
    assert rls._searches[R] is rs
    fresh = RLSynthesis(env, {}, mc, device=0)
    fresh.policy.load_state_dict(other)
    want = [fresh.synth(t, num_searches=R, seed=3) for t in targets]
    rls.synth(targets[0], num_searches=R, seed=3)
    fresh.synth(targets[0], num_searches=R, seed=3)
    assert not np.array_equal(_returns(fresh._searches[R]), before)
    assert np.array_equal(_returns(rs), _returns(fresh._searches[R]))
    assert [str(g) for g in got] == [str(w) for w in want]
