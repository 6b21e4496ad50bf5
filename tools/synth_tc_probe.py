#!/usr/bin/env python
"""Wall time of RolloutSearch.solve_many with the "tensor_core" backend against the one-launch "persistent" (f32 FFMA) backend, alternated
in one process, `rounds` each (median, min, max).  Cases: C5 (Permutation 27q heavy-hex) and C3 (Clifford 8q all-to-all), R rollouts per
target in {100, 1000}, T targets up to 65 536 // R, one launch per case (targets_per_launch = T, as RLSynthesis.solve_many picks it); a
seeded random-weight BasicPolicy of the default shape (512 -> 256, the fused three-layer tensor-core kernel); seeded random targets.  With
random weights almost no rollout succeeds, so almost every rollout runs the whole 128-decision budget.  The two backends round
differently, so their results are not compared; each line gives both success fractions.
Then, per config and batch, a per-decision split from CUDA events over a 128-decision eager search: observe (once per search: the step
writes the next observation itself), policy (qg_policy_tc_forward_bits, and the FFMA policy qg_policy_forward_bits on the same
observations for comparison) and step (qg_search_step_bits).
Lines (JSON): the card (read in the same run), then one per case, then one per split.
    python tools/synth_tc_probe.py [--rounds 3] [--out FILE.jsonl]"""
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

CASES = {100: (1, 16, 148, 655), 1000: (1, 16, 65)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def stats(v):
    v = sorted(v)
    return {"s_median": v[len(v) // 2], "s_min": v[0], "s_max": v[-1]}


def timed_many(rs, states, seed):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = rs.solve_many(states, seed=seed)
    return time.perf_counter() - t0, res


def split(tc, ffma, state, seed, decisions):
    """Mean per-decision times (us) of an eager search on tc's engine: observe once, then decisions x (TC policy, FFMA policy, step)."""
    env = tc.env
    B = tc.B
    with torch.cuda.stream(tc._stream):
        env.set_state_grouped([state] * tc.targets_per_launch, tc.R)
        env.search_begin(seed, 0)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 + 3 * decisions)]
        ev[0].record()
        tc._observe()
        ev[1].record()
        for d in range(decisions):
            tc.handle.forward_bits(tc.obs_bits, probs=tc.probs)
            ev[2 + 3 * d].record()
            ffma.handle.forward_bits(tc.obs_bits, probs=ffma.probs)          # (same observations; its output is not used)
            ev[3 + 3 * d].record()
            env.search_step_bits(tc.probs, tc.obs_bits, num_active=tc.num_active)
            ev[4 + 3 * d].record()
        tc._stream.synchronize()
    pol, ffm, stp = [], [], []
    prev = ev[1]
    for d in range(decisions):
        a, b, c = ev[2 + 3 * d], ev[3 + 3 * d], ev[4 + 3 * d]
        pol.append(prev.elapsed_time(a) * 1e3)
        ffm.append(a.elapsed_time(b) * 1e3)
        stp.append(b.elapsed_time(c) * 1e3)
        prev = c
    mean = lambda v: sum(v) / len(v)
    return {"part": "split", "rollouts": B, "decisions": decisions, "observe_us": ev[0].elapsed_time(ev[1]) * 1e3,
            "policy_tc_us": mean(pol), "policy_ffma_us": mean(ffm), "step_us": mean(stp), "active_after": int(tc.num_active.item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", nargs="+", default=["C5_perm27_heavyhex", "C3_clifford8_full"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("synth_tc_probe needs a CUDA device")
    lines = [{"part": "card", "nvidia_smi": card(), "torch": torch.__version__}]
    print(json.dumps(lines[-1]), flush=True)
    seed = 3
    for name in args.configs:
        kind, n, gs, _ = W.baseline_configs()[name]
        kw = {} if kind == W.PAULI else {"add_inverts": False}
        probe = BatchedEnv(kind, n, gs, 1, add_perms=False, **kw)
        torch.manual_seed(0)
        pol = BasicPolicy(probe.obs_shape(), probe.num_actions(), embedding_size=512, common_layers=(256,))
        all_states = [r.tolist() for r in W.random_targets(kind, n, gs, max(max(t) for t in CASES.values()), 7)]
        for R, Ts in CASES.items():
            for T in Ts:
                states = all_states[:T]
                ss = {b: RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, policy_backend=b, **kw) for b in ("persistent", "tensor_core")}
                for rs in ss.values():
                    rs.solve_many(states, seed=seed)                      # warm-up (module load, graph capture)
                t = {b: [] for b in ss}
                res = {}
                for _ in range(args.rounds):                              # alternating
                    for b, rs in ss.items():
                        dt, res[b] = timed_many(rs, states, seed)
                        t[b].append(dt)
                p, q = stats(t["persistent"]), stats(t["tensor_core"])
                rec = {"part": "case", "config": name, "rollouts_per_target": R, "targets": T, "rollouts_per_launch": R * T, "rounds": args.rounds,
                       "persistent": p, "tensor_core": q, "speedup_median": p["s_median"] / q["s_median"],
                       "decisions": {b: max(r.iterations for r in res[b]) for b in ss},
                       "success_fraction": {b: sum(r.success for r in res[b]) / T for b in ss},
                       "note": "random-weight policy: almost every rollout runs the full 128-decision budget"}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
                if T == Ts[-1] or (R == 100 and T == 16):
                    ffma = RolloutSearch(kind, n, gs, pol, R, targets_per_launch=T, policy_backend="fused", **kw)
                    rec = dict(split(ss["tensor_core"], ffma, states[0], seed, 128), config=name)
                    lines.append(rec)
                    print(json.dumps(rec), flush=True)
                    del ffma
                del ss
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
