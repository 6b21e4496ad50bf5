#!/usr/bin/env python
"""Targets per second of a multi-target search (RolloutSearch.solve_many, one-launch "persistent" backend) against a Python loop of
single-target solve() calls, alternated in one process, `rounds` each.  Cases: C5 (Permutation 27q heavy-hex) and C3 (Clifford 8q
all-to-all), R rollouts per target in {100, 1000}, T targets in {1, 16, 148, 1024}; a seeded random-weight BasicPolicy of the default shape
(512 -> 256); seeded random targets (uniform permutations, Cliffords scrambled by 256 gates).  With random weights almost no rollout
succeeds, so almost every rollout runs the whole 128-decision budget: this measures the search at its full length.  solve_many runs
min(T, 65 536 // R) targets per launch, as RLSynthesis.solve_many does by default.  Every line also checks that both ways return the
same results (key, rollout id, actions) for every target.  Lines (JSON): the card (read in the same run), then one per case.
    python tools/synth_many_probe.py [--rounds 3] [--out FILE.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from qiskit_gym_b200 import BatchedEnv
from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.search import BasicPolicy, RolloutSearch

MAX_ROLLOUTS = 65536


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def targets(kind, n, gs, T, seed):
    rows = W.random_targets(kind, n, gs, T, seed)
    return [r.tolist() for r in rows]


def run_loop(rs, states, R, seed):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = [rs.solve(s, seed=seed, first_rollout_id=t * R) for t, s in enumerate(states)]
    return time.perf_counter() - t0, res


def run_many(rs, states, seed):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = rs.solve_many(states, seed=seed)
    return time.perf_counter() - t0, res


def stats(v):
    v = sorted(v)
    return {"s_median": v[len(v) // 2], "s_min": v[0], "s_max": v[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", nargs="+", default=["C5_perm27_heavyhex", "C3_clifford8_full"])
    ap.add_argument("--rollouts", type=int, nargs="+", default=[100, 1000])
    ap.add_argument("--targets", type=int, nargs="+", default=[1, 16, 148, 1024])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("synth_many_probe needs a CUDA device")
    lines = [{"part": "card", "nvidia_smi": card(), "torch": torch.__version__}]
    print(json.dumps(lines[-1]), flush=True)
    seed = 3
    for name in args.configs:
        kind, n, gs, _ = W.baseline_configs()[name]
        kw = {} if kind == W.PAULI else {"add_inverts": False}
        probe = BatchedEnv(kind, n, gs, 1, add_perms=False, **kw)
        torch.manual_seed(0)
        pol = BasicPolicy(probe.obs_shape(), probe.num_actions(), embedding_size=512, common_layers=(256,))
        all_states = targets(kind, n, gs, max(args.targets), 7)
        for R in args.rollouts:
            single = RolloutSearch(kind, n, gs, pol, R, **kw)
            single.solve(all_states[0], seed=seed)                 # warm-up (module load, scratch growth)
            for T in args.targets:
                states = all_states[:T]
                tpl = min(T, max(1, MAX_ROLLOUTS // R))
                many = RolloutSearch(kind, n, gs, pol, R, targets_per_launch=tpl, **kw)
                many.solve_many(states[:1], seed=seed)            # warm-up
                tl, tm = [], []
                for _ in range(args.rounds):                         # alternating
                    dt, loop_res = run_loop(single, states, R, seed)
                    tl.append(dt)
                    dt, many_res = run_many(many, states, seed)
                    tm.append(dt)
                same = all((a.key, a.rollout_id, a.actions) == (b.key, b.rollout_id, b.actions) for a, b in zip(loop_res, many_res))
                rec = {"part": "case", "config": name, "rollouts_per_target": R, "targets": T, "targets_per_launch": tpl, "rounds": args.rounds,
                       "loop_solve": stats(tl), "solve_many": stats(tm), "same_results": same,
                       "targets_per_s_loop": T / stats(tl)["s_median"], "targets_per_s_many": T / stats(tm)["s_median"],
                       "speedup_median": stats(tl)["s_median"] / stats(tm)["s_median"],
                       "decisions_per_launch_mean": sum(r.iterations for r in many_res) / T, "success_fraction": sum(r.success for r in many_res) / T,
                       "note": "random-weight policy: almost every rollout runs the full 128-decision budget"}
                del many
                lines.append(rec)
                print(json.dumps(rec), flush=True)
            del single
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
