"""Tree reuse between tree-search decisions (MCTSSearch(reuse_tree=True), qg_mcts_reroot / qg_mcts_begin_keep in csrc/qg_mcts.cu).

`reroot` below restates the protocol on per-node lists.  The CPU tests pin the restatement itself on hand-built trees; the GPU tests
hold the device to it: the kernel on hand-built device trees (tree arrays and pool records), and whole searches decision by decision
against CpuTree (tests/test_mcts.py) grown with the pool's own coin draws, so that with add_inverts the tree's child and the rollout
really reach different envs and the search falls back to a fresh tree."""
import types

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests import helpers as H
from tests.test_mcts import CpuTree
from tests.test_search import STREAM_SAMPLE, cpu_pick

f32 = np.float32
STREAM_COIN = 2          # qg_common.cuh: the add_inverts coin
NODE_FIELDS = ("P", "N", "W", "child", "reward", "final")


def reroot_plan(child, count, c, keep):
    """Old ids of the nodes a re-rooted tree keeps, in their new order: the first `keep` members of c's subtree in creation order."""
    member, kept = {c}, []
    for j in range(c, count):
        if len(kept) == keep:
            break
        if j in member:
            kept.append(j)
            member.update(int(x) for x in child[j] if x >= 0)
    return kept


def reroot(tree, a, same_record, keep, fields=NODE_FIELDS):
    """The protocol of qg_mcts_reroot on one tree whose per-node lists are the attributes `fields` (child among them).
    same_record(c): whether node c's env record equals the rollout's.  Returns whether the tree was re-rooted (it is then
    rewritten in place: kept nodes renumbered in creation order, dropped children -1, N / W / P untouched)."""
    if a < 0:
        return False
    c = int(tree.child[0][a])
    if c < 0 or not same_record(c):
        return False
    kept = reroot_plan(tree.child, len(tree.child), c, keep)
    new_id = {o: i for i, o in enumerate(kept)}
    for f in fields:
        setattr(tree, f, [getattr(tree, f)[o] for o in kept])
    tree.child = [np.array([new_id.get(int(x), -1) for x in row], dtype=np.int64) for row in tree.child]
    return True


# ---- the restatement on hand-built trees (CPU) ----------------------------------------------------------------------------------
def hand_tree(parents, A, final=()):
    """Tree with node j > 0 created under parents[j] = (parent, action); N / W / P / reward distinct per entry."""
    n = len(parents) + 1
    t = types.SimpleNamespace()
    t.child = [np.full(A, -1, np.int64) for _ in range(n)]
    for j, (p, a) in enumerate(parents, start=1):
        assert p < j and t.child[p][a] < 0
        t.child[p][a] = j
    t.N = [np.arange(A, dtype=np.int64) + 10 * j for j in range(n)]
    t.W = [np.arange(A, dtype=f32) * f32(0.5) + f32(j) for j in range(n)]
    t.P = [np.full(A, f32(1.0 / (j + 2)), f32) for j in range(n)]
    t.reward = [f32(-0.01 * j) for j in range(n)]
    t.final = [j in final for j in range(n)]
    t.rec = list(range(n))                   # stands for node j's env record
    return t


def check_rerooted(before, after, kept):
    """Prefix closure, id remap, moved payloads, dropped edges keeping N / W."""
    new_id = {o: i for i, o in enumerate(kept)}
    assert kept == sorted(kept)
    for i, o in enumerate(kept):
        for f in ("P", "N", "W"):
            assert np.array_equal(np.asarray(after.__dict__[f][i]), np.asarray(before.__dict__[f][o]))
        assert after.reward[i] == before.reward[o] and after.final[i] == before.final[o] and after.rec[i] == before.rec[o]
        for a, x in enumerate(before.child[o]):
            assert after.child[i][a] == (new_id[x] if x in new_id else -1)
    parent = {int(x): o for o in range(len(before.child)) for x in before.child[o] if x >= 0}
    for o in kept[1:]:
        assert parent[o] in new_id and new_id[parent[o]] < new_id[o]


def _copy(t):
    return types.SimpleNamespace(**{k: list(v) for k, v in t.__dict__.items()})


def test_reroot_chain_overflowing_keep():
    # root -a0-> 1 -a1-> 2 -a1-> 3 ... a chain of 9 nodes under the played child, plus a sibling branch under the root
    parents = [(0, 0), (0, 2)] + [(1, 1)] + [(j, 1) for j in range(3, 10)]
    t = hand_tree(parents, A=3)
    before = _copy(t)
    keep = 4
    assert reroot(t, 0, lambda c: True, keep, NODE_FIELDS + ("rec",))
    kept = reroot_plan(before.child, len(before.child), 1, keep)
    assert kept == [1, 3, 4, 5] and len(t.child) == keep
    check_rerooted(before, t, kept)
    # the last kept node's edge to its dropped child keeps N and W, child -1
    assert t.child[3][1] == -1 and t.N[3][1] == before.N[5][1] and t.W[3][1] == before.W[5][1]


def test_reroot_branching_prefix_in_creation_order():
    rng = np.random.default_rng(3)
    A = 4
    for trial in range(50):
        parents = []
        for j in range(1, 30):
            while True:
                p, a = int(rng.integers(j)), int(rng.integers(A))
                if all(q != (p, a) for q in parents):
                    parents.append((p, a))
                    break
        t = hand_tree(parents, A)
        before = _copy(t)
        a = int(rng.integers(A))
        c = int(t.child[0][a])
        keep = int(rng.integers(1, 12))
        assert reroot(t, a, lambda c: True, keep, NODE_FIELDS + ("rec",)) == (c >= 0)
        if c >= 0:
            kept = reroot_plan(before.child, len(before.child), c, keep)
            assert kept[0] == c and len(t.child) == len(kept) <= keep
            check_rerooted(before, t, kept)


def test_reroot_missing_child_final_child_and_record_mismatch():
    t = hand_tree([(0, 0), (1, 0)], A=2, final={1})
    same = lambda c: True
    assert not reroot(_copy(t), 1, same, 3, NODE_FIELDS + ("rec",))            # no child under action 1
    assert not reroot(_copy(t), -1, same, 3, NODE_FIELDS + ("rec",))           # rollout already final: nothing played
    assert not reroot(_copy(t), 0, lambda c: False, 3, NODE_FIELDS + ("rec",))  # the rollout reached another env
    f = _copy(t)
    assert reroot(f, 0, same, 3, NODE_FIELDS + ("rec",))                       # final child: kept with its final flag
    assert f.final[0] and f.rec[0] == 1 and len(f.child) == 2


# ---- the device against the restatement -----------------------------------------------------------------------------------------
class ReuseTree(CpuTree):
    """CpuTree whose children are stepped with the pool's coin (seed 0, logical tree index, the parent's step counter), which
    tracks each node's step counter and inversion parity (the record's FL_INVERTED bit, which the oracle does not expose)."""

    def __init__(self, root_env, prior, A, c_puct, index, tick, inv, coins):
        super().__init__(root_env, prior, A, c_puct)
        self.index, self.coins = index, coins
        self.tick, self.inv = [tick], [inv]

    def expand(self, parent, a):
        coin = (orc.philox_draw(0, self.index, self.tick[parent], STREAM_COIN) >> 31) if self.coins else None
        env = self.envs[parent].clone()
        env.step(a, coin=coin)
        self.child[parent][a] = len(self.envs)
        self.envs.append(env)
        self.N.append(np.zeros(self.A, np.int64)); self.W.append(np.zeros(self.A, f32)); self.child.append(np.full(self.A, -1, np.int64))
        self.P.append(None)
        self.reward.append(f32(env.reward())); self.final.append(env.is_final())
        self.tick.append(self.tick[parent] + 1); self.inv.append(self.inv[parent] ^ int(bool(coin)))
        return len(self.envs) - 1


def env_key(env, inv):
    """What an env record holds, seen through the oracle."""
    return (env.raw_state().tobytes(), inv, env.depth(), tuple(env.counts()), np.float32(env.reward()).tobytes(), env.success(), env.is_final())


@pytest.mark.gpu
@pytest.mark.parametrize("name,deterministic", [("C1_perm_grid3", False), ("clifford3_allgates", True), ("lf5_line_swap", False),
                                                ("lf5_line_swap", True), ("pauli3_line", False)])
def test_reuse_matches_cpu_restatement(name, deterministic):
    """Decision by decision: root visit weights, chosen actions, reused flags and final states of the device search with reuse equal
    those of CpuTree re-rooted by `reroot`; add_inverts is on wherever the env has it."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy

    kind, n, gs, kw = H.config_table()[name]
    kw = dict(kw, add_perms=False)
    coins = kind != H.PAULI
    if coins:
        kw["add_inverts"] = True
    R, S, decisions, seed, first, cp = 37, 12, 9, 21, 300, 1.5
    K = S + 1
    A = len(gs)
    tgt_env = orc.OracleEnv(kind, n, gs, difficulty=4, **kw)
    tgt_env.reset(seed=4, env_id=0)
    if kind == H.PAULI:
        t = H.random_targets(kind, n, gs, 1, 3, scramble=3, num_rotations=2)
        target = t[0, : H.payload_lengths(kind, n, t)[0]].tolist()
    else:
        target = tgt_env.raw_state().astype(np.int64).tolist()
    torch.manual_seed(1)
    ekw = dict(max_depth=10, **kw)
    probe = orc.OracleEnv(kind, n, gs, **ekw)
    pol = BasicPolicy(probe.obs_shape(), A, embedding_size=32, common_layers=(16,))
    with torch.no_grad():
        for prm in pol.action.parameters():
            prm.mul_(50.0)              # peaked priors: the simulations pile up under few children, so kept subtrees outgrow K
    ms = MCTSSearch(kind, n, gs, pol, R, S, C=cp, reuse_tree=True, **ekw)
    assert ms.NC == 2 * S + 1
    rec = {}
    ms.hook = lambda kind_, d, s, p, v: rec.__setitem__((kind_, d, s), (p.cpu().numpy().copy(), None if v is None else v.cpu().numpy().copy()))
    ms.env.set_state(target)
    ms.env.search_begin(seed, first)
    refs = []
    for b in range(R):
        r = orc.OracleEnv(kind, n, gs, **ekw)
        r.set_state(target)
        refs.append(r)
    ticks, rinv = np.zeros(R, np.int64), np.zeros(R, np.int64)
    trees = [None] * R
    expected_reused = np.zeros(R, np.uint8)
    stats = dict(reused=0, fresh_after_step=0, pruned=0)
    for d in range(decisions):
        w_gpu = ms.decide(d).cpu().numpy()
        assert np.array_equal(ms.reused.cpu().numpy(), expected_reused), d
        ms.env.search_step(ms.weights, deterministic=deterministic, obs=False, chosen=ms.chosen)
        got = ms.chosen.cpu().numpy()
        root_prior = rec[("root", d, -1)][0]
        for b, r in enumerate(refs):
            tree = trees[b] if expected_reused[b] else ReuseTree(r.clone(), root_prior[b], A, cp, b, int(ticks[b]), int(rinv[b]), coins)
            for s in range(S):
                p, v = rec[("leaf", d, s)]
                path, parent, a = tree.select()
                if a >= 0:
                    new = tree.expand(parent, a)
                    tree.P[new] = p[b].astype(f32)
                    tree.backup(path, f32(0) if tree.final[new] else v[b])
                else:
                    tree.backup(path, f32(0))
            w = tree.root_weights()
            assert np.array_equal(w.view(np.uint32), w_gpu[b].view(np.uint32)), (d, b, w, w_gpu[b])
            if r.is_final():
                assert got[b] == -1
                expected_reused[b] = 0
                continue
            raw = orc.philox_draw(seed, first + b, int(ticks[b]), STREAM_SAMPLE)
            act = cpu_pick(w, raw, deterministic)
            assert got[b] == act, (d, b)
            coin = (orc.philox_draw(seed, first + b, int(ticks[b]), STREAM_COIN) >> 31) if coins else None
            r.step(act, coin=coin)
            ticks[b] += 1
            rinv[b] ^= int(bool(coin))
            key = env_key(r, int(rinv[b]))
            c = int(tree.child[0][act])
            members = len(reroot_plan(tree.child, len(tree.child), c, len(tree.child))) if c >= 0 else 0
            ok = reroot(tree, act, lambda c: env_key(tree.envs[c], tree.inv[c]) == key, K, NODE_FIELDS + ("envs", "tick", "inv"))
            stats["pruned"] += int(ok and members > K)
            expected_reused[b] = 1 if ok else 0
            stats["reused" if ok else "fresh_after_step"] += 1
            trees[b] = tree
    assert stats["reused"] > R and stats["pruned"] > 0, stats
    if coins:
        assert stats["fresh_after_step"] > R // 2, stats          # coin mismatches really occurred
    for b in range(R):
        assert np.array_equal(ms.env.get_state(b), refs[b].raw_state())


def _random_parents(rng, count, A, chain_from=None):
    parents = []
    for j in range(1, count):
        if chain_from is not None and j > chain_from:
            parents.append((j - 1, int(rng.integers(A))))
            continue
        while True:
            p, a = int(rng.integers(j)), int(rng.integers(A))
            if all(q != (p, a) for q in parents):
                parents.append((p, a))
                break
    return parents


@pytest.mark.gpu
def test_reroot_kernel_on_hand_built_trees():
    """qg_mcts_reroot on device trees built by hand (random shapes, chains that overflow keep_nodes, a missing child, a final child,
    records that differ from the rollout's) against `reroot`: tree arrays and the moved pool records, read back per slot."""
    from qiskit_gym_b200.engine import BatchedEnv
    from qiskit_gym_b200.mcts import TreeArrays

    kind, n, gs, kw = H.config_table()["C2_lf8_line"]
    A, NC, keep, R = len(gs), 25, 13, 40
    rng = np.random.default_rng(11)
    targets = H.random_targets(kind, n, gs, R * NC + R, 5, scramble=12)
    dev = torch.device("cuda", 0)
    pool = BatchedEnv(kind, n, gs, R * NC, device=0, add_inverts=False, add_perms=False, track_solution=False)
    roll = BatchedEnv(kind, n, gs, R, device=0, add_inverts=False, add_perms=False)
    pool.set_state(targets[: R * NC])
    ta = TreeArrays(R, NC, A, dev)
    trees, chosen, roll_rows = [], np.full(R, -1, np.int32), []
    for i in range(R):
        count = int(rng.integers(2, NC + 1))
        t = hand_tree(_random_parents(rng, count, A, chain_from=1 if i % 3 == 0 else None), A, final={1} if i % 7 == 3 else ())
        t.N = [rng.integers(0, 50, A) for _ in range(count)]
        t.W = [rng.standard_normal(A).astype(f32) for _ in range(count)]
        t.P = [rng.random(A).astype(f32) for _ in range(count)]
        t.reward = [f32(rng.standard_normal()) for _ in range(count)]
        t.rec = [i * NC + j for j in range(count)]                 # the pool slot whose target node j holds
        trees.append(t)
        root_actions = np.nonzero(t.child[0] >= 0)[0]
        if i % 11 == 5:
            a = -1                                                  # the rollout was final: nothing played
        elif i % 3 == 0:
            a = int(np.nonzero(t.child[0] == 1)[0][0])             # into the chain below node 1
        elif i % 5 == 2:
            a = int(rng.integers(A))                                # often an action without a child
        else:
            a = int(rng.choice(root_actions))
        chosen[i] = a
        c = int(t.child[0][a]) if a >= 0 else -1
        # the rollout holds node c's env, except in every fourth tree
        roll_rows.append(targets[i * NC + c] if (c >= 0 and i % 4 != 1) else targets[R * NC + i])
    with torch.no_grad():
        for i, t in enumerate(trees):
            cnt = len(t.child)
            ta.prior[i, :cnt] = torch.from_numpy(np.stack(t.P))
            ta.visits[i, :cnt] = torch.from_numpy(np.stack(t.N).astype(np.int32))
            ta.value_sum[i, :cnt] = torch.from_numpy(np.stack(t.W))
            ta.child[i, :cnt] = torch.from_numpy(np.stack(t.child).astype(np.int32))
            ta.node_reward[i, :cnt] = torch.from_numpy(np.array(t.reward, f32))
            ta.node_final[i, :cnt] = torch.from_numpy(np.array(t.final, np.uint8))
            ta.node_count[i] = cnt
    roll.set_state(np.stack(roll_rows))
    pool_before = [pool.get_state(k) for k in range(R * NC)]
    before = {k: getattr(ta, k).cpu().numpy().copy() for k in ("prior", "visits", "value_sum", "child", "node_reward", "node_final", "node_count")}
    chosen_d = torch.from_numpy(chosen).to(dev)
    reused = torch.zeros(R, dtype=torch.uint8, device=dev)
    ta.reroot(pool, roll, chosen_d, keep, reused)
    torch.cuda.synchronize()
    got = {k: getattr(ta, k).cpu().numpy() for k in before}
    ru = reused.cpu().numpy()
    seen = dict(reused=0, fresh=0, pruned=0)
    for i, t in enumerate(trees):
        a = int(chosen[i])
        roll_state = roll.get_state(i)
        same = lambda c: np.array_equal(pool_before[i * NC + c], roll_state)
        c = int(t.child[0][a]) if a >= 0 else -1
        if c >= 0 and len(reroot_plan(t.child, len(t.child), c, NC)) > keep:
            seen["pruned"] += 1
        ok = reroot(t, a, same, keep, NODE_FIELDS + ("rec",))
        assert ru[i] == (1 if ok else 0), i
        if not ok:
            seen["fresh"] += 1
            for k in before:
                assert np.array_equal(got[k][i], before[k][i]), (i, k)
            continue
        seen["reused"] += 1
        cnt = len(t.child)
        assert got["node_count"][i] == cnt
        assert np.array_equal(got["prior"][i, :cnt].view(np.uint32), np.stack(t.P).view(np.uint32))
        assert np.array_equal(got["visits"][i, :cnt], np.stack(t.N))
        assert np.array_equal(got["value_sum"][i, :cnt].view(np.uint32), np.stack(t.W).view(np.uint32))
        assert np.array_equal(got["child"][i, :cnt], np.stack(t.child))
        assert np.array_equal(got["node_reward"][i, :cnt].view(np.uint32), np.array(t.reward, f32).view(np.uint32))
        assert np.array_equal(got["node_final"][i, :cnt], np.array(t.final, np.uint8))
        for j in range(cnt):                        # pool slot i * NC + j now holds the env of old slot t.rec[j]
            assert np.array_equal(pool.get_state(i * NC + j), pool_before[t.rec[j]]), (i, j)
    assert seen["reused"] > 5 and seen["fresh"] > 5 and seen["pruned"] > 0, seen


@pytest.mark.gpu
@pytest.mark.parametrize("sims", [12, 130])
def test_graph_replay_equals_eager_with_reuse(sims):
    """With reuse the captured decision (reroot inside the whole-decision graph, or inside the root graph beyond 128 simulations) leaves
    the same visit weights and reused flags, bit for bit, as the launch-by-launch search; with add_inverts off every rollout that played
    an action keeps its tree."""
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C2_lf8_line"]
    torch.manual_seed(1)
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,))
    R = 96
    tarr = H.random_targets(kind, n, gs, R, 3, scramble=6)
    out = {}
    for graph in (False, True):
        ms = MCTSSearch(kind, n, gs, pol, R, sims, max_depth=16, add_inverts=False, use_cuda_graph=graph, reuse_tree=True)
        ms.env.set_state(tarr)
        ms.env.search_begin(5, 0)
        w, ru = [], []
        for d in range(4):
            prev = ms.chosen.clone()
            w.append(ms.decide(d).clone())
            ru.append(ms.reused.clone())
            assert torch.equal(ms.reused.bool(), prev >= 0), d
            ms.env.search_step(ms.weights, deterministic=True, obs=False, chosen=ms.chosen)
        out[graph] = (w, ru)
        if graph:
            assert ms._graphs is not None
    assert sum(int(r.sum()) for r in out[False][1]) > R
    for a, b in zip(out[False][0], out[True][0]):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    for a, b in zip(out[False][1], out[True][1]):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_reuse_solve_finds_shallow_targets():
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy
    kind, n, gs, kw = H.config_table()["C1_perm_grid3"]
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,))
    ms = MCTSSearch(kind, n, gs, pol, 64, 16, max_depth=6, add_inverts=False, reuse_tree=True)
    tgt = orc.OracleEnv(kind, n, gs, difficulty=2, add_inverts=False, add_perms=False)
    solved = 0
    for trial in range(3):
        tgt.reset(seed=trial, env_id=0)
        state = tgt.raw_state().astype(np.int64).tolist()
        res = ms.solve(state, deterministic=False, seed=trial)
        if res.actions is not None:
            solved += 1
            chk = orc.OracleEnv(kind, n, gs, add_inverts=False, add_perms=False)
            chk.set_state(state)
            for a in res.actions:
                chk.step(a)
            assert chk.success()
    assert solved >= 2


@pytest.mark.gpu
def test_rlsynthesis_reuse_tree_api():
    """reuse_tree is a separate cached search; reuse_tree=False is the search of a call without it; reuse needs a tree search;
    synth with reuse returns circuits that implement the target."""
    import os
    from qiskit_gym_b200.rl import RLSynthesis
    models = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models")
    rls = RLSynthesis.from_config_json(os.path.join(models, "lf_5_line.json"), os.path.join(models, "lf_5_line.pt"))
    n = rls.env_config["num_qubits"]
    edges = [tuple(q) for g, q in rls.env_config["gateset"] if g.lower() == "cx"]
    rng = np.random.default_rng(2)
    with pytest.raises(ValueError):
        rls.solve(rls.env.get_state(np.eye(n, dtype=np.uint8)), num_searches=4, reuse_tree=True)
    with pytest.raises(ValueError):
        rls.synth(np.eye(n, dtype=np.uint8), num_searches=4, reuse_tree=True)
    solved = 0
    for t in range(4):
        M = np.eye(n, dtype=np.uint8)
        for _ in range(6):
            a, b = edges[int(rng.integers(len(edges)))]
            M[b] ^= M[a]
        st = rls.env.get_state(M)
        base = rls.solve(st, deterministic=False, num_searches=16, num_mcts_searches=8, seed=t)
        assert rls.solve(st, deterministic=False, num_searches=16, num_mcts_searches=8, seed=t, reuse_tree=False) == base
        circ = rls.synth(M, deterministic=False, num_searches=16, num_mcts_searches=8, seed=t, reuse_tree=True)
        if circ is None:
            continue
        solved += 1
        G = np.eye(n, dtype=np.uint8)
        for g, (a, b) in circ:
            if g.lower() == "cx":
                G[b] ^= G[a]
            else:
                G[[a, b]] = G[[b, a]]
        assert np.array_equal(G, M)
    assert solved >= 3
    keys = [k for k in rls._searches if k[0] == "mcts"]
    assert sorted(k[-1] for k in keys) == [False, True]
    assert rls._searches[keys[0]] is not rls._searches[keys[1]]
