#!/usr/bin/env python
"""Tree reuse between tree-search decisions (MCTSSearch(reuse_tree=True)) on one GPU: what it costs and what it buys.

Part "time": per-decision wall time of the device tree search with and without reuse, alternated in one process, medians of `rounds`, at C1
(Permutation 3x3 grid) and C3 (Clifford 8q all-to-all), R rollouts in {96, 1024}, S simulations in {16, 100}; a seeded random-weight
BasicPolicy (64 -> 32), seeded random targets (difficulty 64), add_inverts off (so every tree that played an action is kept), `decisions`
decisions after one warm-up decision, CUDA graphs on (the default).  The same case also times qg_mcts_reroot alone: CUDA events around
each of `launches` launches, each on the trees and pool records of a real decision restored beforehand (restore outside the events).

Part "quality": the reference's trained checkpoints (tests/golden/models) in the reference's `mcts_100` setting (one rollout, deterministic,
RLSynthesis.solve with num_mcts_searches = S), S in {4, 16, 100}, with and without reuse, on `targets` seeded targets per checkpoint
scrambled at the smallest difficulty of a ladder where greedy decoding (num_mcts_searches = 0) fails on more than 10 % of 64 calibration
targets.  Success rate, mean solution length of the successes, and the reuse rate (re-rooted trees / decisions after a played action).
The checkpoints' envs keep add_inverts on, as they were trained.

Lines (JSON): the card (read in the same run), then one per case.
    python tools/mcts_reuse_probe.py [--parts time quality] [--out FILE.jsonl]"""
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
from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.mcts import MCTSSearch
from qiskit_gym_b200.search import BasicPolicy

MODELS = os.path.join(ROOT, "tests", "golden", "models")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def decisions_time(ms, tarr, decisions, seed):
    """Seconds per decision over `decisions` decisions after one warm-up decision of a fresh search (as solve runs them)."""
    env = ms.env
    env.set_state(tarr)
    env.search_begin(seed, 0)
    ms.chosen.fill_(-1)
    ms._fresh = True
    ms.decide(0)
    env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reused = 0
    for d in range(1, decisions + 1):
        ms.decide(d)
        env.search_step(ms.weights, deterministic=False, obs=False, chosen=ms.chosen)
        reused += int(ms.reused.sum())
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / decisions, reused / (decisions * ms.R)


def reroot_time(ms, launches):
    """CUDA-event time of qg_mcts_reroot alone on the trees of the search's last decision (restored before every launch)."""
    tree, keep = ms.tree, ms.NC - ms.S
    names = ("prior", "visits", "value_sum", "child", "node_reward", "node_final", "node_count", "path_node")
    saved = {k: getattr(tree, k).clone() for k in names}
    ms.pool.snapshot()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    for i in range(launches):
        for k in names:
            getattr(tree, k).copy_(saved[k])
        ms.pool.restore()
        ev[i][0].record()
        tree.reroot(ms.pool, ms.env, ms.chosen, keep, ms.reused)
        ev[i][1].record()
    torch.cuda.synchronize()
    us = sorted(a.elapsed_time(b) * 1e3 for a, b in ev[launches // 10:])          # (the first tenth warms up)
    return {"reroot_us_median": us[len(us) // 2], "reroot_us_min": us[0], "reroot_us_max": us[-1], "reroot_reused": int(ms.reused.sum())}


def part_time(args, out):
    for name in ("C1_perm_grid3", "C3_clifford8_full"):
        kind, n, gs, _ = W.baseline_configs()[name]
        for R in (96, 1024):
            tarr = W.random_targets(kind, n, gs, R, 11, scramble=64)
            for S in (16, 100):
                torch.manual_seed(0)
                probe = orc.OracleEnv(kind, n, gs, add_inverts=False, add_perms=False)
                pol = BasicPolicy(probe.obs_shape(), len(gs), embedding_size=64, common_layers=(32,))
                ms = {r: MCTSSearch(kind, n, gs, pol, R, S, max_depth=128, add_inverts=False, reuse_tree=r) for r in (False, True)}
                t = {False: [], True: []}
                rate = None
                for _ in range(args.rounds):
                    for r in (False, True):
                        s, rr = decisions_time(ms[r], tarr, args.decisions, seed=5)
                        t[r].append(s)
                        if r:
                            rate = rr
                line = {"part": "time", "config": name, "R": R, "S": S, "decisions": args.decisions, "rounds": args.rounds,
                        "decision_ms_no_reuse": sorted(t[False])[len(t[False]) // 2] * 1e3, "decision_ms_reuse": sorted(t[True])[len(t[True]) // 2] * 1e3,
                        "reuse_rate": rate, **reroot_time(ms[True], args.launches)}
                line["reroot_share_of_reuse_decision"] = line["reroot_us_median"] * 1e-3 / line["decision_ms_reuse"]
                out(line)
                del ms
                torch.cuda.empty_cache()


def part_quality(args, out):
    from qiskit_gym_b200.rl import RLSynthesis, _ENV_KINDS
    for name in ("perm_square_3x3", "lf_5_line", "clifford_3q_custom"):
        rls = RLSynthesis.from_config_json(os.path.join(MODELS, name + ".json"), os.path.join(MODELS, name + ".pt"), device=0)
        cfg = rls.env_config
        kind, n = _ENV_KINDS[rls.env.cls_name], cfg["num_qubits"]
        gs = [(g, tuple(q)) for g, q in cfg["gateset"]]

        def targets(difficulty, count, base):
            e = orc.OracleEnv(kind, n, gs, difficulty=difficulty, add_inverts=False, add_perms=False)
            out_ = []
            for t in range(count):
                e.reset(seed=base + t, env_id=0)
                out_.append(e.raw_state().astype(np.int64).tolist())
            return out_

        chosen_d, greedy = None, None
        for d in (2, 4, 8, 12, 16, 24, 32, 48, 64, 96, 128):
            ok = sum(rls.solve(s, deterministic=True, num_searches=1, seed=0) is not None for s in targets(d, 64, 10_000))
            chosen_d, greedy = d, ok / 64
            if greedy < 0.9:
                break
        states = targets(chosen_d, args.targets, 0)
        g_ok = [rls.solve(s, deterministic=True, num_searches=1, seed=0) for s in states]
        out({"part": "quality", "checkpoint": name, "difficulty": chosen_d, "greedy_calibration_success": greedy,
             "S": 0, "reuse_tree": False, "targets": len(states), "success_rate": sum(a is not None for a in g_ok) / len(states),
             "mean_length": float(np.mean([len(a) for a in g_ok if a is not None])) if any(a is not None for a in g_ok) else None})
        for S in (4, 16, 100):
            for reuse in (False, True):
                ms = rls._mcts(1, S, 1.41, reuse)
                tally = {"decisions": 0, "reused": 0}

                def hook(kind_, d, s, p, v, ms=ms, tally=tally):
                    if kind_ == "root" and d > 0 and int(ms.chosen[0]) >= 0:
                        tally["decisions"] += 1
                        tally["reused"] += int(ms.reused[0])
                ms.hook = hook if reuse else None           # (the hook runs decisions launch by launch: same results as the graphs)
                res = [ms.solve(s, deterministic=True, seed=0).actions for s in states]
                ms.hook = None
                good = [a for a in res if a is not None]
                out({"part": "quality", "checkpoint": name, "difficulty": chosen_d, "S": S, "C": 1.41, "reuse_tree": reuse, "targets": len(states),
                     "success_rate": len(good) / len(states), "mean_length": float(np.mean([len(a) for a in good])) if good else None,
                     "reuse_rate": (tally["reused"] / tally["decisions"]) if reuse and tally["decisions"] else None})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", nargs="+", default=["time", "quality"])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--decisions", type=int, default=8)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--targets", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mcts_reuse_probe needs a CUDA device")
    fh = open(args.out, "w") if args.out else None

    def out(line):
        print(json.dumps(line), flush=True)
        if fh:
            fh.write(json.dumps(line) + "\n")
            fh.flush()
    out({"part": "card", "nvidia_smi": card(), "torch": torch.__version__})
    if "time" in args.parts:
        part_time(args, out)
    if "quality" in args.parts:
        part_quality(args, out)


if __name__ == "__main__":
    main()
