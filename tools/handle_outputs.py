#!/usr/bin/env python
"""Fixed-seed outputs of every consumer of a device policy handle, for comparing two source trees bit for bit:
RolloutSearch.solve_many on each backend, MCTSSearch.solve with and without reuse_tree (fused and PyTorch policy), and
RolloutCollector.collect / collect_packed.  Weight updates happen only where both trees refresh the handle in place (the
"tensor_core" search, the packed collector).

    python tools/handle_outputs.py --tree DIR --out FILE.pt     # imports qiskit_gym_b200 from DIR
    python tools/handle_outputs.py --compare A.pt B.pt          # exit code 1 unless every output is identical
"""
import argparse
import os
import sys


def _update(pol):
    import torch
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(-1.5)


def _results(res):
    return [(r.actions, r.key, r.rollout_id, r.success, r.iterations, r.rollouts) for r in res]


def _rollout(ro):
    fields = ("obs", "obs_bits", "actions", "policy_actions", "logp", "values", "rewards", "dones", "successes", "valid", "advantages",
              "returns", "twist")
    return {f: getattr(ro, f).detach().cpu().clone() for f in fields if getattr(ro, f) is not None}


def run(tree):
    sys.path.insert(0, os.path.abspath(tree))
    import torch
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200 import workloads as W
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.mcts import MCTSSearch
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch

    out = {}
    kind, n, gs, kw = W.baseline_configs()["C3_clifford8_full"]
    targets = [t.tolist() for t in W.random_targets(kind, n, gs, 12, 5, scramble=6)]
    for backend in ("torch", "fused", "persistent", "tensor_core"):
        torch.manual_seed(1)
        pol = BasicPolicy([2 * n, 2 * n], len(gs))
        rs = RolloutSearch(kind, n, gs, pol, 500, max_depth=64, policy_backend=backend, targets_per_launch=4, **kw)
        out[f"solve_many/{backend}"] = _results(rs.solve_many(targets, seed=3))
        out[f"solve_many/{backend}/det"] = _results(rs.solve_many(targets, deterministic=True, seed=3))
        if backend == "tensor_core":
            _update(pol)
            out[f"solve_many/{backend}/updated"] = _results(rs.solve_many(targets, seed=3))
    for backend in ("fused", "torch"):
        for reuse in (False, True):
            torch.manual_seed(2)
            pol = BasicPolicy([2 * n, 2 * n], len(gs), embedding_size=128, common_layers=(64,))
            ms = MCTSSearch(kind, n, gs, pol, 64, 16, max_depth=32, policy_backend=backend, reuse_tree=reuse, **kw)
            out[f"mcts/{backend}/reuse={reuse}"] = _results([ms.solve(t, seed=s) for s, t in enumerate(targets[:4])])
    for packed in (False, True):
        env = BatchedEnv(kind, n, gs, 8192, difficulty=6, add_perms=True, **kw)
        torch.manual_seed(3)
        pol = BasicPolicy(env.obs_shape(), env.num_actions())
        col = RolloutCollector(env, pol, seed=11, first_env_id=7)
        collect = col.collect_packed if packed else col.collect
        for it in range(3):
            out[f"collect/packed={packed}/{it}"] = _rollout(collect(16))
        if packed:
            _update(pol)
            out["collect/packed=True/updated"] = _rollout(collect(16))
    torch.cuda.synchronize()
    return out


def same(a, b):
    import torch
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return isinstance(b, (list, tuple)) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return a == b


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree")
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        a, b = (torch.load(p, weights_only=False) for p in args.compare)
        bad = sorted(set(a) ^ set(b)) + [k for k in a if k in b and not same(a[k], b[k])]
        print(f"{len(a)} outputs compared; differing: {bad or 'none'}")
        sys.exit(1 if bad else 0)
    torch.save(run(args.tree), args.out)


if __name__ == "__main__":
    main()
