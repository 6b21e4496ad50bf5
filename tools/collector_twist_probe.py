#!/usr/bin/env python
"""Twists on the packed tensor-core collector, measured.  Two parts, one JSON line each (plus the card it ran on):
  collect : RolloutCollector.collect_packed (CUDA graph) at C3 (C3_clifford8_full, add_perms=True, BasicPolicy 512/256), untwisted and
            twisted collectors alternating in the same process, `rounds` timed rollouts each; us per decision, CUDA events.
  ppo     : one PPO iteration split into collect / update / eval (host clock around device-synchronised work) for matmul_precision
            "f32" (dense PyTorch collector) and "tensor_core" (collect_packed) at num_episodes 1 024 and 65 536.
    python tools/collector_twist_probe.py [--envs 65536] [--decisions 32] [--rounds 5] [--out FILE.jsonl]"""
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
from qiskit_gym_b200.collector import RolloutCollector
from qiskit_gym_b200.ppo import PPO
from qiskit_gym_b200.search import BasicPolicy


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def part_collect(B, T, rounds):
    kind, n, gateset, _ = W.baseline_configs()["C3_clifford8_full"]
    torch.manual_seed(0)
    pol = BasicPolicy([2 * n, 2 * n], len(gateset), embedding_size=512, common_layers=(256,)).cuda()
    cols = {}
    for name, tw in (("untwisted", False), ("twisted", True)):
        env = BatchedEnv(kind, n, gateset, B, device=0, difficulty=64, depth_slope=2, max_depth=128, add_perms=True, add_inverts=False)
        cols[name] = RolloutCollector(env, pol, use_twists=tw, seed=0)
        for _ in range(3):                                  # eager, capture, first replay
            cols[name].collect_packed(T)
    torch.cuda.synchronize()
    us = {k: [] for k in cols}
    for _ in range(rounds):
        for name, col in cols.items():                      # alternating
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            col.collect_packed(T)
            e1.record()
            torch.cuda.synchronize()
            us[name].append(1e3 * e0.elapsed_time(e1) / T)
    out = {"part": "collect", "config": "C3_clifford8_full add_perms", "envs": B, "decisions": T, "num_twists": cols["twisted"].num_twists}
    for k, v in us.items():
        v = sorted(v)
        out[k] = {"us_per_decision_median": v[len(v) // 2], "us_per_decision_min": v[0], "us_per_decision_max": v[-1],
                  "env_steps_per_s_median": B / (v[len(v) // 2] * 1e-6)}
    out["twist_overhead"] = out["twisted"]["us_per_decision_median"] / out["untwisted"]["us_per_decision_median"] - 1.0
    return out


def part_ppo(episodes, precision, iters):
    kind, n, gateset, _ = W.baseline_configs()["C3_clifford8_full"]
    torch.manual_seed(0)
    pol = BasicPolicy([2 * n, 2 * n], len(gateset), embedding_size=512, common_layers=(256,))
    cfg = {"collecting": {"num_episodes": episodes}, "training": {"num_epochs": 10},
           "evals": {"ppo_deterministic": {"num_episodes": 100}}}
    ppo = PPO(kind, n, gateset, pol, cfg, device=0, seed=1, matmul_precision=precision, difficulty=4, add_perms=True, add_inverts=False)
    T = ppo._episode_steps()
    rows = []

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    for it in range(iters + 2):                             # the first two iterations warm up (and capture the collector's graph)
        ro, tc = timed(lambda: ppo.collector.collect_packed(T) if ppo.tensor_core else ppo.collector.collect(T))
        st, tu = timed(lambda: ppo.update(ro))
        _, te = timed(lambda: ppo.evaluate("ppo_deterministic"))
        if it >= 2:
            rows.append((tc, tu, te, st["samples"]))
    med = lambda i: sorted(r[i] for r in rows)[len(rows) // 2]        # noqa: E731
    return {"part": "ppo", "config": "C3_clifford8_full add_perms difficulty 4", "matmul_precision": precision, "num_episodes": episodes,
            "decisions": T, "num_epochs": 10, "iterations_timed": len(rows), "collect_s": med(0), "update_s": med(1), "eval_s": med(2),
            "samples": rows[-1][3]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--decisions", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ppo-iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collector_twist_probe needs a CUDA device")
    lines = [{"part": "card", "nvidia_smi": card(), "torch": torch.__version__}]
    lines.append(part_collect(args.envs, args.decisions, args.rounds))
    print(json.dumps(lines[-1]), flush=True)
    for episodes in (1024, 65536):
        for precision in ("f32", "tensor_core"):
            lines.append(part_ppo(episodes, precision, args.ppo_iters))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
