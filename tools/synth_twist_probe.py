#!/usr/bin/env python
"""The twisted rollout search (RolloutSearch(use_twists=True)) against the untwisted one.
1. Time per decision, twisted and untwisted alternated in one process, `rounds` each (median, min, max): the one-launch "persistent" search at
   C1 (Permutation 3x3 grid, K = 8), C3 (Clifford 8q all-to-all, K = 40 320) and C5 (Permutation 27q heavy-hex) with R = 1 000 rollouts of
   one target, and the "tensor_core" solve_many at C3 with T = 65 targets x R = 1 000.  A seeded random-weight BasicPolicy of the default
   shape (512 -> 256): almost no rollout succeeds, so every search runs the whole 128-decision budget; time per decision = wall time of the
   search (ending in a device synchronise) / decisions taken.
2. Search quality on the three reference checkpoints under tests/golden/models: per checkpoint and difficulty, 256 seeded targets (the
   oracle env's reset at that difficulty), num_searches = 100, sampled, twisted and untwisted (RLSynthesis.solve_many): success rate and
   mean solution length of the solved targets.
Lines (JSON): the card (name, power limit, max SM clock; read in the same run), then one per case.
    python tools/synth_twist_probe.py [--rounds 3] [--out FILE.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from oracle import oracle as orc
from qiskit_gym_b200 import BatchedEnv
from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.rl import RLSynthesis
from qiskit_gym_b200.search import BasicPolicy, RolloutSearch

MODELS = os.path.join(ROOT, "tests", "golden", "models")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def stats(v):
    v = sorted(v)
    return {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}


def timed(rs, states, seed):
    """(seconds per decision, decisions) of one search: solve for one target, solve_many for several."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = rs.solve(states[0], seed=seed) if rs.targets_per_launch == 1 else rs.solve_many(states, seed=seed)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    its = max(r.iterations for r in (res if isinstance(res, list) else [res]))
    return dt / its, its


def timing(name, backend, R, T, rounds, lines):
    kind, n, gs, _ = W.baseline_configs()[name]
    kw = {"add_inverts": False}
    probe = BatchedEnv(kind, n, gs, 1, add_perms=False, **kw)
    torch.manual_seed(0)
    pol = BasicPolicy(probe.obs_shape(), probe.num_actions(), embedding_size=512, common_layers=(256,))
    states = [r.tolist() for r in W.random_targets(kind, n, gs, T, 7)]
    ss = {tw: RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, policy_backend=backend, use_twists=tw, **kw) for tw in (False, True)}
    for rs in ss.values():
        timed(rs, states, 3)                                      # warm-up (module load, graph capture)
    t = {tw: [] for tw in ss}
    its = {}
    for _ in range(rounds):                                       # alternating
        for tw, rs in ss.items():
            dt, its[tw] = timed(rs, states, 3)
            t[tw].append(dt * 1e6)
    u, w = stats(t[False]), stats(t[True])
    rec = {"part": "time", "config": name, "backend": backend, "rollouts_per_target": R, "targets": T, "rounds": rounds, "num_twists": ss[True].num_twists,
           "act_table_bytes": int(ss[True].act_table.numel() * 4), "untwisted_us_per_decision": u, "twisted_us_per_decision": w,
           "twisted_over_untwisted_median": w["median"] / u["median"], "decisions": {"untwisted": its[False], "twisted": its[True]},
           "note": "random-weight default-shape policy: every rollout runs the 128-decision budget"}
    lines.append(rec)
    print(json.dumps(rec), flush=True)


def quality(model, difficulty, lines, count=256, R=100):
    rls = RLSynthesis.from_config_json(os.path.join(MODELS, model + ".json"), os.path.join(MODELS, model + ".pt"))
    kind, n, gs, kw = rls._env_args(add_perms=False)
    kw = {k: v for k, v in kw.items() if k != "difficulty"}
    gs = [(g, tuple(q)) for g, q in gs]
    tgt = orc.OracleEnv(kind, n, gs, difficulty=difficulty, **kw)
    states = []
    for i in range(count):
        tgt.reset(seed=1000 + i, env_id=0)
        states.append(tgt.raw_state().astype(np.int64).tolist())
    rec = {"part": "quality", "model": model, "difficulty": difficulty, "targets": count, "num_searches": R, "deterministic": False}
    for tw in (False, True):
        acts = rls.solve_many(states, num_searches=R, seed=11, use_twists=tw)
        ok = [a for a in acts if a is not None]
        rec["twisted" if tw else "untwisted"] = {"success_rate": len(ok) / count, "mean_length": (sum(map(len, ok)) / len(ok)) if ok else None}
    rec["num_twists"] = rls._search(R, count, use_twists=True).num_twists
    lines.append(rec)
    print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("synth_twist_probe needs a CUDA device")
    lines = [{"part": "card", "nvidia_smi": card(), "torch": torch.__version__}]
    print(json.dumps(lines[-1]), flush=True)
    for name in ("C1_perm_grid3", "C3_clifford8_full", "C5_perm27_heavyhex"):
        timing(name, "persistent", 1000, 1, args.rounds, lines)
    timing("C3_clifford8_full", "tensor_core", 1000, 65, args.rounds, lines)
    for model in ("perm_square_3x3", "lf_5_line", "clifford_3q_custom"):
        for difficulty in (8, 32):
            quality(model, difficulty, lines)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
