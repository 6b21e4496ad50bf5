#!/usr/bin/env python
"""The PPO update on the tensor cores, measured.  At C3 (C3_clifford8_full, add_perms=True, BasicPolicy 512/256, difficulty 4, 10 epochs),
num_episodes 1 024 and 65 536, on one packed tensor-core rollout per size.  Lines (JSON, plus the card, read in the same run):
  profile : torch.profiler (CUDA activities) over one PPO.update per update_precision: the device-time share of GEMM kernels, of the
            project's tcgen05 kernels (qg::tc), of Adam and of everything else (the loss's elementwise ops, gathers, reductions).
  update  : PPO.update timed (host clock around device-synchronised work) for update_precision "f32" and "tensor_core", alternated in one
            process, `rounds` each; policy and optimiser state restored before every run, so both do the same work.
  phases  : one full-batch optimiser step split with CUDA events into the training forward, the backward (loss included) and Adam.
    python tools/ppo_update_probe.py [--rounds 3] [--out FILE.jsonl]"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from qiskit_gym_b200 import workloads as W
from qiskit_gym_b200.collector import unpack_bits
from qiskit_gym_b200.ppo import PPO
from qiskit_gym_b200.search import BasicPolicy


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # (the probe still runs; the line says why the card is unknown)
        return f"unknown ({e})"


def make(episodes):
    kind, n, gateset, _ = W.baseline_configs()["C3_clifford8_full"]
    torch.manual_seed(0)
    pol = BasicPolicy([2 * n, 2 * n], len(gateset), embedding_size=512, common_layers=(256,))
    cfg = {"collecting": {"num_episodes": episodes}, "training": {"num_epochs": 10}}
    ppo = PPO(kind, n, gateset, pol, cfg, device=0, seed=1, matmul_precision="tensor_core", update_precision="tensor_core", difficulty=4,
              add_perms=True, add_inverts=False)
    ro = ppo.collector.collect_packed(ppo._episode_steps())
    return ppo, ro


def run_update(ppo, ro, precision, state):
    ppo.policy.load_state_dict(state[0])
    ppo.opt.load_state_dict(state[1])
    ppo.update_tc = precision == "tensor_core"
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st = ppo.update(ro)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, st


def classify(name):
    n = name.lower()
    if "qg::tc" in n or "k_tc_" in n:
        return "tcgen05"
    if "gemm" in n or "cutlass" in n or "xmma" in n or "cublas" in n or "sm90_" in n or "sm100_" in n or "nvjet" in n:
        return "gemm"
    if "adam" in n or "multi_tensor_apply" in n:           # torch.optim.Adam's foreach kernels
        return "adam"
    return "other"


def profile(ppo, ro, precision, state):
    from torch.profiler import ProfilerActivity, profile as tprof
    ppo.policy.load_state_dict(state[0])
    ppo.opt.load_state_dict(state[1])
    ppo.update_tc = precision == "tensor_core"
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        ppo.update(ro)
        torch.cuda.synchronize()
    tot, by = 0.0, {}
    top = []
    for e in prof.key_averages():
        t = float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
        if t <= 0 or e.key.startswith("ProfilerStep"):
            continue
        if getattr(e, "device_type", None) is not None and "CUDA" not in str(e.device_type):
            continue
        c = classify(e.key)
        by[c] = by.get(c, 0.0) + t
        tot += t
        top.append((t, e.key[:90], c))
    top.sort(reverse=True)
    return {"device_us": tot, "share": {k: v / tot for k, v in by.items()} if tot else {}, "top": [[round(t, 1), k, c] for t, k, c in top[:8]]}


def phases(ppo, ro, precision, state, reps=3):
    """One full-batch optimiser step (the first epoch's), CUDA events between forward, loss + backward and Adam; median of reps."""
    ppo.policy.load_state_dict(state[0])
    ppo.opt.load_state_dict(state[1])
    t = ppo.cfg["training"]
    idx = ro.valid.reshape(-1).nonzero(as_tuple=False).squeeze(1)
    bits = ro.obs_bits.reshape(-1, ro.obs_bits.shape[-1])[idx]
    act, logp_old = ro.policy_actions.reshape(-1)[idx], ro.logp.reshape(-1)[idx]
    adv, ret = ro.advantages.reshape(-1)[idx], ro.returns.reshape(-1)[idx]
    obs = unpack_bits(bits, ro.obs_size).reshape((-1,) + tuple(ppo.env.obs_shape())) if precision == "f32" else None
    clip = float(t["clip_ratio"])
    out = []
    for _ in range(reps + 1):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ppo.opt.zero_grad(set_to_none=True)
        ev[0].record()
        if precision == "f32":
            logits, value = ppo.policy(obs)
        else:
            logits, value = ppo._train_policy(bits.shape[0]).forward_train(ppo.policy, bits)
        ev[1].record()
        logp_all = torch.log_softmax(logits.float(), dim=-1)
        logp = logp_all.gather(1, act[:, None]).squeeze(1)
        ratio = torch.exp(logp - logp_old)
        pi_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * adv).mean()
        v_loss = torch.nn.functional.mse_loss(value.float().reshape(-1), ret)
        entropy = -(logp_all.exp() * logp_all).sum(-1).mean()
        (pi_loss + float(t["vf_coef"]) * v_loss - float(t["ent_coef"]) * entropy).backward()
        ev[2].record()
        ppo.opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        out.append([ev[i].elapsed_time(ev[i + 1]) for i in range(3)])
    out = out[1:]
    med = lambda i: sorted(r[i] for r in out)[len(out) // 2]        # noqa: E731
    return {"forward_ms": med(0), "loss_and_backward_ms": med(1), "adam_ms": med(2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--episodes", type=int, nargs="+", default=[1024, 65536])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_update_probe needs a CUDA device")
    lines = [{"part": "card", "nvidia_smi": card(), "torch": torch.__version__}]
    print(json.dumps(lines[-1]), flush=True)
    for episodes in args.episodes:
        ppo, ro = make(episodes)
        state = (copy.deepcopy(ppo.policy.state_dict()), copy.deepcopy(ppo.opt.state_dict()))
        base = {"config": "C3_clifford8_full add_perms difficulty 4", "num_episodes": episodes, "num_epochs": 10,
                "samples": int(ro.valid.sum().item())}
        for precision in ("f32", "tensor_core"):                # warm-up: every shape, the training handle, cuBLAS' choices
            run_update(ppo, ro, precision, state)
        for precision in ("f32", "tensor_core"):
            lines.append(dict(base, part="profile", update_precision=precision, **profile(ppo, ro, precision, state)))
            print(json.dumps(lines[-1]), flush=True)
        times = {"f32": [], "tensor_core": []}
        for _ in range(args.rounds):
            for precision in times:                              # alternating
                times[precision].append(run_update(ppo, ro, precision, state)[0])
        rec = dict(base, part="update", rounds=args.rounds)
        for precision, v in times.items():
            v = sorted(v)
            rec[precision] = {"update_s_median": v[len(v) // 2], "update_s_min": v[0], "update_s_max": v[-1]}
        rec["speedup"] = rec["f32"]["update_s_median"] / rec["tensor_core"]["update_s_median"]
        lines.append(rec)
        print(json.dumps(lines[-1]), flush=True)
        for precision in ("f32", "tensor_core"):
            lines.append(dict(base, part="phases", update_precision=precision, **phases(ppo, ro, precision, state)))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
