#!/usr/bin/env python
"""Persistent searches (qg_search_run) on C5 with 1000 rollouts: for ncu captures of k_search_fused and for splitting a
decision's time between the policy network and the env step (a tiny policy leaves only the step + barriers).  Prints the
kernel's own time (CUDA events) next to the wall time of the whole solve() call."""
import sys
import numpy as np
import torch
sys.path.insert(0, ".")
from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.search import BasicPolicy, RolloutSearch

kind, n, gs, kw = W.baseline_configs()["C5_perm27_heavyhex"]
rng = np.random.Generator(np.random.PCG64(1))
for emb, common in ((512, (256,)), (32, ())):
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=emb, common_layers=common)
    rs = RolloutSearch(kind, n, gs, pol, 1000, max_depth=128, add_inverts=False, policy_backend="persistent")
    for i in range(3):
        r = rs.solve(rng.permutation(n).astype(np.int64).tolist(), seed=i)
    env = rs.env
    env.set_state(rng.permutation(n).astype(np.int64).tolist())
    env.search_begin(7, 0)
    env.observe_bits(rs.obs_bits)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    env.search_run(rs.handle, rs.obs_bits, rs.probs, 128, decisions=rs._decisions)
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1)
    print(emb, common, r.iterations, "solve() %.3f ms wall; kernel %.3f ms = %.1f us per decision" % (r.seconds * 1e3, k_ms, k_ms * 1e3 / 128))
