#!/usr/bin/env python
"""The tree search on the tensor-core policy (MCTSSearch(policy_backend="tensor_core")) against the f32 fused one ("fused") on one GPU: where
the tensor cores start to pay, what AlphaZero self-play gains at scale, and what the arithmetic does to solution quality.

Part "time": per-decision wall time (host clock around decisions that end in a device synchronise) of "fused" and "tensor_core", alternated
in one process, medians of `rounds`, at C1 (Permutation 3x3 grid), C3 (Clifford 8q all-to-all) and C5 (Permutation 27q heavy hex), R trees in
{128, 1 024, 4 096, 8 192}, S simulations in {16, 100}; a seeded random-weight policy of the reference's default shape (obs -> 512 -> 256 ->
A + 1: 256 -> 512 -> 256 -> A + 1 at C3), seeded random targets (difficulty 64), add_inverts off, fresh trees, `decisions` decisions after one
warm-up decision, CUDA graphs on (the default).  A point whose engines or trees cannot be allocated is reported as skipped.  Then per config
and S the crossover: the smallest R of the sweep from which "tensor_core" is faster at every larger R (null: slower at every R tried).

Part "az": one AlphaZero iteration (self-play + update, 4 epochs) at C3 with 4 096 episodes and S = 16, matmul_precision "f32" and
"tensor_core", alternated, medians of `rounds` after one warm-up iteration each, difficulty 2, the default-shape policy.

Part "quality": the reference's trained checkpoints (tests/golden/models) in the reference's `mcts_100` setting (one rollout, deterministic,
100 simulations, C = 1.41) through RLSynthesis.solve(..., matmul_precision="f32" / "tensor_core"), on `targets` seeded targets per checkpoint
at difficulty 128 (where greedy decoding of these checkpoints still solves every calibration target: tools/mcts_twist_probe.py).  Success
rate and mean solution length of the successes.  The checkpoints' envs keep add_inverts on, as they were trained.

Lines (JSON): the card (read in the same run), then one per case.
    python tools/mcts_tc_probe.py [--parts time az quality] [--out FILE.jsonl]"""
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
from qiskit_gym_b200.mcts import MCTSSearch
from qiskit_gym_b200.search import BasicPolicy
from tools.mcts_reuse_probe import MODELS, card, decisions_time

BACKENDS = ("fused", "tensor_core")


def median(v):
    return sorted(v)[len(v) // 2]


def default_policy(kind, n, gs, seed=0):
    torch.manual_seed(seed)
    probe = orc.OracleEnv(kind, n, gs, add_inverts=False, add_perms=False)
    return BasicPolicy(probe.obs_shape(), len(gs), embedding_size=512, common_layers=(256,))


def part_time(args, out):
    for name in ("C1_perm_grid3", "C3_clifford8_full", "C5_perm27_heavyhex"):
        kind, n, gs, _ = W.baseline_configs()[name]
        pol = default_policy(kind, n, gs)
        for S in (16, 100):
            ratios = {}
            for R in (128, 1024, 4096, 8192):
                tarr = W.random_targets(kind, n, gs, R, 11, scramble=64)
                ms = {}
                try:
                    for b in BACKENDS:
                        ms[b] = MCTSSearch(kind, n, gs, pol, R, S, max_depth=128, add_inverts=False, policy_backend=b)
                except (torch.cuda.OutOfMemoryError, RuntimeError) as e:
                    out({"part": "time", "config": name, "R": R, "S": S, "skipped": f"pool and tree arrays do not fit: {e}"[:300]})
                    ms = None
                    torch.cuda.empty_cache()
                    continue
                t = {b: [] for b in BACKENDS}
                for _ in range(args.rounds):
                    for b in BACKENDS:
                        t[b].append(decisions_time(ms[b], tarr, args.decisions, seed=5)[0])
                line = {"part": "time", "config": name, "R": R, "S": S, "decisions": args.decisions, "rounds": args.rounds,
                        "decision_ms_fused": median(t["fused"]) * 1e3, "decision_ms_tensor_core": median(t["tensor_core"]) * 1e3}
                line["tensor_core_over_fused"] = line["decision_ms_tensor_core"] / line["decision_ms_fused"]
                ratios[R] = line["tensor_core_over_fused"]
                out(line)
                del ms
                torch.cuda.empty_cache()
            Rs = sorted(ratios)
            cross = next((R for i, R in enumerate(Rs) if all(ratios[r] < 1.0 for r in Rs[i:])), None)
            out({"part": "crossover", "config": name, "S": S, "R_tried": Rs, "tensor_core_faster_from_R": cross,
                 "note": "tensor_core slower below this R" if cross is not None else "tensor_core slower at every R tried (crossover above)"})


def part_az(args, out):
    from qiskit_gym_b200.ppo import AlphaZero
    kind, n, gs, _ = W.baseline_configs()["C3_clifford8_full"]
    E, S = 4096, 16
    cfg = {"collecting": {"num_episodes": E, "num_mcts_searches": S, "C": 1.41}, "training": {"num_epochs": 4}}
    az = {}
    for prec in ("f32", "tensor_core"):
        az[prec] = AlphaZero(kind, n, gs, default_policy(kind, n, gs), cfg, device=0, seed=1, matmul_precision=prec, add_inverts=False)
        az[prec].difficulty = 2
        az[prec].iterate()
    t, rec = {"f32": [], "tensor_core": []}, {}
    for _ in range(args.rounds):
        for prec in az:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rec[prec] = az[prec].iterate()
            torch.cuda.synchronize()
            t[prec].append(time.perf_counter() - t0)
    out({"part": "az", "config": "C3_clifford8_full", "episodes": E, "S": S, "epochs": 4, "difficulty": 2, "rounds": args.rounds,
         "steps_per_iteration": az["f32"]._episode_steps(), "iteration_ms_f32": median(t["f32"]) * 1e3,
         "iteration_ms_tensor_core": median(t["tensor_core"]) * 1e3, "tensor_core_over_f32": median(t["tensor_core"]) / median(t["f32"]),
         "samples": {p: r["samples"] for p, r in rec.items()}})


def part_quality(args, out):
    from qiskit_gym_b200.rl import RLSynthesis, _ENV_KINDS
    S, difficulty = 100, 128
    for name in ("perm_square_3x3", "lf_5_line", "clifford_3q_custom"):
        rls = RLSynthesis.from_config_json(os.path.join(MODELS, name + ".json"), os.path.join(MODELS, name + ".pt"), device=0)
        cfg = rls.env_config
        kind, n = _ENV_KINDS[rls.env.cls_name], cfg["num_qubits"]
        gs = [(g, tuple(q)) for g, q in cfg["gateset"]]
        e = orc.OracleEnv(kind, n, gs, difficulty=difficulty, add_inverts=False, add_perms=False)
        states = []
        for t in range(args.targets):
            e.reset(seed=t, env_id=0)
            states.append(e.raw_state().astype(np.int64).tolist())
        for prec in ("f32", "tensor_core"):
            t0 = time.perf_counter()
            res = [rls.solve(s, deterministic=True, num_searches=1, num_mcts_searches=S, C=1.41, seed=0, matmul_precision=prec) for s in states]
            good = [a for a in res if a is not None]
            out({"part": "quality", "checkpoint": name, "difficulty": difficulty, "S": S, "C": 1.41, "matmul_precision": prec,
                 "targets": len(states), "success_rate": len(good) / len(states),
                 "mean_length": float(np.mean([len(a) for a in good])) if good else None, "seconds": time.perf_counter() - t0})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", nargs="+", default=["time", "az", "quality"])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--decisions", type=int, default=4)
    ap.add_argument("--targets", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mcts_tc_probe needs a CUDA device")
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
