#!/usr/bin/env python
"""The twisted tree search (MCTSSearch(use_twists=True)) and twisted AlphaZero self-play on one GPU: what the twists cost and what they do
to solution quality.

Part "time": per-decision wall time (host clock around decisions that end in a device synchronise) of the device tree search twisted and
untwisted, alternated in one process, medians of `rounds`, at C1 (Permutation 3x3 grid, K = 8), C3 (Clifford 8q all-to-all, K = 40 320) and
C5 (Permutation 27q heavy hex), R rollouts in {96, 1024}, S simulations in {16, 100}, with and without tree reuse; a seeded random-weight
BasicPolicy (64 -> 32), seeded random targets (difficulty 64), add_inverts off, `decisions` decisions after one warm-up decision, CUDA graphs
on (the default).  For each config and R (S = 16, no reuse) the twisted node-observation kernel (qg_mcts_observe_twisted) is timed alone:
CUDA events around each of `launches` root-pass and leaf-pass launches on the records of a real decision.

Part "az": one AlphaZero iteration (self-play + update) at C1, twisted and untwisted, alternated, medians of `rounds` after one warm-up
iteration each (256 episodes, 16 simulations, 4 epochs).

Part "quality": the reference's trained checkpoints (tests/golden/models) in the reference's `mcts_100` setting (one rollout,
deterministic, 100 simulations), twisted and untwisted, on `targets` seeded targets per checkpoint scrambled at the smallest difficulty of a
ladder where greedy decoding fails on more than 10 % of 64 calibration targets (as tools/mcts_reuse_probe.py).  Success rate and mean
solution length of the successes.  The checkpoints' envs keep add_inverts on, as they were trained.

Lines (JSON): the card (read in the same run), then one per case.
    python tools/mcts_twist_probe.py [--parts time az quality] [--out FILE.jsonl]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from oracle import oracle as orc
from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.mcts import MCTSSearch, observe_twisted
from qiskit_gym_b200.search import BasicPolicy
from tools.mcts_reuse_probe import MODELS, card, decisions_time


def median(v):
    return sorted(v)[len(v) // 2]


def observe_time(ms, launches):
    """CUDA-event time of qg_mcts_observe_twisted alone, root pass and leaf pass, on the search's last decision (the leaf pass reads
    the slots of its last simulation; the evaluation counter is restored before every leaf launch)."""
    out = {}
    for leaf in (False, True):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
        saved = ms.eval_index.clone()
        for i in range(launches):
            ms.eval_index.copy_(saved)
            ev[i][0].record()
            if leaf:
                observe_twisted(ms.env, ms.pool, ms.dst, ms.act, ms.search_key, ms.eval_index, ms.qperm_table, ms.leaf_bits, ms.leaf_twist)
            else:
                observe_twisted(ms.env, None, None, None, ms.search_key, ms.eval_index, ms.qperm_table, ms.root_bits, ms.root_twist)
            ev[i][1].record()
        torch.cuda.synchronize()
        us = sorted(a.elapsed_time(b) * 1e3 for a, b in ev[launches // 10:])          # (the first tenth warms up)
        p = "observe_leaf" if leaf else "observe_root"
        out.update({p + "_us_median": us[len(us) // 2], p + "_us_min": us[0], p + "_us_max": us[-1]})
    return out


def part_time(args, out):
    for name in ("C1_perm_grid3", "C3_clifford8_full", "C5_perm27_heavyhex"):
        kind, n, gs, _ = W.baseline_configs()[name]
        for R in (96, 1024):
            tarr = W.random_targets(kind, n, gs, R, 11, scramble=64)
            for S in (16, 100):
                for reuse in (False, True):
                    torch.manual_seed(0)
                    probe = orc.OracleEnv(kind, n, gs, add_inverts=False, add_perms=False)
                    pol = BasicPolicy(probe.obs_shape(), len(gs), embedding_size=64, common_layers=(32,))
                    ms = {tw: MCTSSearch(kind, n, gs, pol, R, S, max_depth=128, add_inverts=False, reuse_tree=reuse, use_twists=tw) for tw in (False, True)}
                    t = {False: [], True: []}
                    for _ in range(args.rounds):
                        for tw in (False, True):
                            t[tw].append(decisions_time(ms[tw], tarr, args.decisions, seed=5)[0])
                    line = {"part": "time", "config": name, "K": ms[True].num_twists, "R": R, "S": S, "reuse_tree": reuse, "decisions": args.decisions,
                            "rounds": args.rounds, "decision_ms_untwisted": median(t[False]) * 1e3, "decision_ms_twisted": median(t[True]) * 1e3}
                    line["twisted_over_untwisted"] = line["decision_ms_twisted"] / line["decision_ms_untwisted"]
                    if S == 16 and not reuse:
                        line.update(observe_time(ms[True], args.launches))
                    out(line)
                    del ms
                    torch.cuda.empty_cache()


def part_az(args, out):
    from qiskit_gym_b200.ppo import AlphaZero
    kind, n, gs, _ = W.baseline_configs()["C1_perm_grid3"]
    cfg = {"collecting": {"num_episodes": 256, "num_mcts_searches": 16, "C": 1.41}, "training": {"num_epochs": 4}}
    az = {}
    for tw in (False, True):
        torch.manual_seed(0)
        pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(64,))
        az[tw] = AlphaZero(kind, n, gs, pol, cfg, device=0, seed=1, use_twists=tw)
        az[tw].difficulty = 4
        az[tw].iterate()
    t = {False: [], True: []}
    for _ in range(args.rounds):
        for tw in (False, True):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rec = az[tw].iterate()
            torch.cuda.synchronize()
            t[tw].append(time.perf_counter() - t0)
    out({"part": "az", "config": "C1_perm_grid3", "episodes": 256, "S": 16, "epochs": 4, "difficulty": 4, "rounds": args.rounds,
         "steps_per_iteration": az[True]._episode_steps(), "iteration_ms_untwisted": median(t[False]) * 1e3, "iteration_ms_twisted": median(t[True]) * 1e3,
         "twisted_over_untwisted": median(t[True]) / median(t[False]), "last_samples": rec["samples"]})


def part_quality(args, out):
    from qiskit_gym_b200.rl import RLSynthesis, _ENV_KINDS
    S = 100
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
        k_, n_, gs_, kw = rls._env_args()
        kw.pop("add_perms", None)
        searches = {False: rls._mcts(1, S, 1.41), True: MCTSSearch(k_, n_, gs_, rls.policy, 1, S, C=1.41, device=rls.device, use_twists=True, **kw)}
        for tw in (False, True):
            t0 = time.perf_counter()
            res = [searches[tw].solve(s, deterministic=True, seed=0).actions for s in states]
            good = [a for a in res if a is not None]
            out({"part": "quality", "checkpoint": name, "difficulty": chosen_d, "greedy_calibration_success": greedy, "S": S, "C": 1.41,
                 "use_twists": tw, "K": searches[True].num_twists, "targets": len(states), "success_rate": len(good) / len(states),
                 "mean_length": float(np.mean([len(a) for a in good])) if good else None, "seconds": time.perf_counter() - t0})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", nargs="+", default=["time", "az", "quality"])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--decisions", type=int, default=8)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--targets", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mcts_twist_probe needs a CUDA device")
    fh = open(args.out, "w") if args.out else None

    def out(line):
        print(json.dumps(line), flush=True)
        if fh:
            fh.write(json.dumps(line) + "\n")
            fh.flush()
    out({"part": "card", "nvidia_smi": card(), "torch": torch.__version__})
    if "time" in args.parts:
        part_time(args, out)
    if "az" in args.parts:
        part_az(args, out)
    if "quality" in args.parts:
        part_quality(args, out)


if __name__ == "__main__":
    main()
