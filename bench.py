#!/usr/bin/env python
"""bench.py — batched env-steps/sec of the fused CUDA step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this engine (under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on host cores

A "step" is one episode pass over the batch: every one of the B environments per GPU (default 65 536,
BASELINE.json configs[2]: CliffordGym 8q all-to-all {H,S,CX}) is restored to its synthetic target and stepped
T = max_depth = 128 times from a resident int32[T][B] action stream; every env-step materialises its dense float
observation, mask, reward, done and success in HBM.  `value` plays the stream with one qg_replay launch per episode
(`per_step_launch` reports the same episode as T single-step launches); `e2e` is the episode through the host-buffer
C-ABI call qg_replay_host (actions H2D, reward/done/success D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

# SURVEY.md §8(d): algorithmic bytes per env-step (fp32 obs, u8 mask, i32 action, f32 reward, u8 done,
# packed state + metrics read and written once).
ALGO_BYTES = {"C1_perm_grid3": 449, "C2_lf8_line": 375, "C3_clifford8_full": 1249, "C4_pauli10_line": 2377, "C5_perm27_heavyhex": 3225}
# of which the packed state + metrics record, read and written once per LAUNCH (2*(S_state + S_metrics)): a replay launch of T env-steps moves
# it once, not T times, so its algorithmic bytes are T*(ALGO - STATE) + STATE per env
STATE_BYTES = {"C1_perm_grid3": 104, "C2_lf8_line": 96, "C3_clifford8_full": 144, "C4_pauli10_line": 264, "C5_perm27_heavyhex": 272}
# dram__bytes_read.sum + dram__bytes_write.sum of one replay launch, from the committed ncu --set full capture (profiles/), keyed by
# (config, envs per GPU, env-steps per launch); None where no capture exists.
TRAFFIC_BYTES_PER_LAUNCH = {
    # profiles/r2_v44_<config>_ncu.txt (ncu --set full of one k_step nsteps=128 replay launch per config, 65 536 envs, this round's final kernels,
    # one observation slab per step): dram__bytes_read.sum + dram__bytes_write.sum.  Within 1 % of the algorithmic bytes (the launch's last dirty
    # lines are still in the 126 MB L2 when the counters stop): no wasted re-reads, and nothing absorbed by L2 either.
    ("C1_perm_grid3", 65536, 128): 38864896 + 2847544000,
    ("C2_lf8_line", 65536, 128): 38106880 + 2293921000,
    ("C3_clifford8_full", 65536, 128): 40289792 + 9224168000,
    ("C4_pauli10_line", 65536, 128): 46339840 + 17687305000,
    ("C5_perm27_heavyhex", 65536, 128): 44766720 + 24731291000,
}
METRIC = "batched env-steps/sec (CliffordGym 8q all-to-all {H,S,CX})"
UNIT = "env-steps/s"


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3_clifford8_full")
    ap.add_argument("--envs", type=int, default=65536, help="environments per GPU")
    ap.add_argument("--episode-steps", type=int, default=128)
    ap.add_argument("--add-inverts", type=int, default=0)
    ap.add_argument("--cpu-sample-envs", type=int, default=0, help="envs in the CPU baseline sample (0 = calibrate to ~15 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-per-step", action="store_true", help="skip the one-launch-per-env-step leg (profiling runs)")
    ap.add_argument("--no-synth", action="store_true", help="skip the synth-search leg (BASELINE.json configs[4])")
    ap.add_argument("--no-packed", action="store_true", help="skip the packed-bit observation leg (qg_replay_bits)")
    ap.add_argument("--no-collector", action="store_true", help="skip the policy-in-the-loop collector leg (collector.RolloutCollector)")
    ap.add_argument("--synth-rollouts", type=int, default=1000, help="num_searches per GPU of the synth leg")
    ap.add_argument("--synth-searches", type=int, default=5, help="timed searches of the synth leg")
    ap.add_argument("--obs-buffers", type=int, default=0, help="slabs of the observation / mask ring a launch rotates over: 0 = automatic (> 2x L2 in total)")
    ap.add_argument("--tile-envs", type=int, default=0, help="qg_config.tile_envs of the env-step legs: 0 = automatic, 16 or 32 (A/B runs)")
    ap.add_argument("--synth-all-backends", action="store_true", help="also time the two-kernel and PyTorch-policy searches")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed episode returned as DIR/<name>.npy "
                                                          "(float32; a fixed sample of environments, under 64 MB in all)")
    args = ap.parse_args(argv)
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA engine's outputs (--impl ours)")
    return args


def workload(args):
    from qiskit_gym_b200 import workloads as W
    kind, n, gateset, kw = W.baseline_configs()[args.config]
    return kind, n, gateset, dict(kw)


def episode_inputs(args, envs, rank=0):
    """The synthetic episode one rank plays, a function of the command line and the rank only (seeded per rank so that shards differ
    but are reproducible): set_state targets int64[envs, payload], actions int32[T, envs] and, with add_inverts, coins uint8[T, envs]."""
    from qiskit_gym_b200 import workloads as W
    kind, n, gateset, _ = workload(args)
    T = args.episode_steps
    targets = W.random_targets(kind, n, gateset, envs, 20261017 + 3 + 1000 * rank, scramble=256)
    rng = np.random.Generator(np.random.PCG64(20261017 + rank))
    actions = W.random_actions(rng, T, envs, len(gateset))
    coins = rng.integers(0, 2, size=(T, envs)).astype(np.uint8) if (args.add_inverts and kind != W.PAULI) else None
    return targets, actions, coins


DUMP_BYTES = 60 << 20          # what --dump-outputs writes, .npy headers aside: under 64 MB


def dump_outputs(out_dir, obs_ring, mask_ring, reward, done, success):
    """Writes what the last replayed episode returned, as float32 .npy files: obs [steps, S, obs_size] and mask [steps, S, A] of the
    env-steps still in the ring (all T with the default ring, otherwise the last ones, oldest first), reward / done / success [T, S].
    The S environments are np.random.default_rng(0).choice(B, S, replace=False) in ascending order, the whole batch where it fits."""
    import torch
    nbuf, B, obs_size = obs_ring.shape
    T, A = reward.shape[0], mask_ring.shape[2]
    steps = min(nbuf, T)
    S = min(B, DUMP_BYTES // (4 * (steps * (obs_size + A) + 3 * T)))
    envs = torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, S, replace=False))).to(obs_ring.device)
    slots = torch.tensor([t % nbuf for t in range(T - steps, T)], device=obs_ring.device)
    out = {"obs": obs_ring.index_select(1, envs).index_select(0, slots), "mask": mask_ring.index_select(1, envs).index_select(0, slots),
           "reward": reward.index_select(1, envs), "done": done.index_select(1, envs), "success": success.index_select(1, envs)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def config_json(args, n_gpus):
    """The workload description: a function of the command line only, so that this arm and `--impl reference` print the same dict."""
    c = {
        "workload": f"{args.config}: BASELINE.json config, {args.envs} envs per GPU x {args.episode_steps} env-steps per step "
                    f"(set_state targets: identity scrambled by 256 random gates; uniform random actions; add_inverts={bool(args.add_inverts)}, "
                    "add_perms=False, track_solution=True, default MetricsWeights)",
        "envs_per_gpu": args.envs, "env_steps_per_step": args.episode_steps, "n_gpus": n_gpus,
        "l2_policy": "one observation / mask slab per env-step of a launch (every step's observation is kept: nothing a launch writes is overwritten "
                     "while it could still sit in the 126 MB L2, so all of it reaches DRAM); the ring is shorter only where it would exceed 64 GB, "
                     "and never shorter than 3x L2",
    }
    return c


# ------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline leg (the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------------
def cpu_run(args, envs, steps=1, warmup=0, threads=None):
    from oracle import oracle as orc
    from qiskit_gym_b200 import workloads as W
    kind, n, gateset, kw = workload(args)
    threads = threads or (os.cpu_count() or 1)
    pk = dict(kw)
    if kind != W.PAULI:
        pk["add_inverts"] = bool(args.add_inverts)
    cfg = orc.make_config(kind, n, gateset, add_perms=False, **pk)
    T = args.episode_steps
    targets, actions, coins = episode_inputs(args, envs)
    lens = W.payload_lengths(kind, n, targets)
    times = []
    for i in range(warmup + steps):
        sec, _ = orc.bench(cfg, targets, lens, actions, coins=coins, threads=threads)
        if i >= warmup:
            times.append(sec)
    tot = sum(times)
    return {"value": envs * T * steps / tot, "seconds": tot, "threads": threads, "envs": envs, "T": T}


def calibrate_cpu_envs(args, target_seconds, threads):
    probe = cpu_run(args, envs=max(64, 16 * threads), threads=threads)
    rate = probe["value"]
    envs = int(rate * target_seconds / args.episode_steps)
    return max(256, min(envs // 64 * 64, 1 << 20))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    envs = args.cpu_sample_envs or args.envs          # the same batch as the GPU arm: one step = envs x episode_steps env-steps
    r = cpu_run(args, envs, steps=args.steps, warmup=args.warmup, threads=threads)
    sample = f"{envs} envs x {args.episode_steps} env-steps per step, oracle C++ port of the Rust core (step+observe+masks+reward+is_final per env-step), {threads} host threads"
    line = {
        "impl": "reference", "metric": METRIC if args.config == "C3_clifford8_full" else f"batched env-steps/sec ({args.config})",
        "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * r["seconds"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (byte-per-bit GF(2)) + f32 reward", "data": "synthetic",
        "config": config_json(args, args.gpus),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200 import workloads as W

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from qiskit_gym_b200._lib import lib as _qg_lib
    _qg_lib().qg_bind_thread_to_device(local)          # the thread that drives the engine runs on the GPU's NUMA node (no-op where sysfs hides the topology)
    if world > 1:
        # whatever NCCL_DEBUG level the box sets (the version banner included) goes to a file: stdout carries the JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/qg_bench_nccl.%h.%p.log")
        dist.init_process_group("nccl", device_id=dev)

    kind, n, gateset, kw = workload(args)
    B, T, K, Wm = args.envs, args.episode_steps, args.steps, max(args.warmup, 0)
    A = len(gateset)
    pk = dict(kw)
    if kind != W.PAULI:
        pk["add_inverts"] = bool(args.add_inverts)
    env = BatchedEnv(kind, n, gateset, B, device=local, max_depth=T, add_perms=False, tile_envs=args.tile_envs, **pk)
    obs_size = int(np.prod(env.obs_shape()))
    targets, actions_h, coins_h = episode_inputs(args, B, rank)
    env.set_state(targets)
    env.snapshot()
    actions = torch.from_numpy(actions_h).to(dev)
    coins = None if coins_h is None else torch.from_numpy(coins_h).to(dev)
    # observation / mask ring: one slab per env-step of an episode, so that a launch never rewrites a line that may still be in L2 (with a short
    # ring and few tiles in flight the L2 absorbs part of the rewrites and the launch "beats" the DRAM bandwidth: profiles/r2_v26_pair_ab.txt)
    obs_bytes = B * obs_size * 4
    nbuf = min(T, max(int(np.ceil(3 * 126e6 / max(obs_bytes, 1))) + 1, int(64e9 // max(obs_bytes + B * A, 1))))
    nbuf = max(2, nbuf)
    if args.obs_buffers > 0:
        nbuf = args.obs_buffers
    obs_ring = torch.empty((nbuf, B, obs_size), dtype=torch.float32, device=dev)
    mask_ring = torch.empty((nbuf, B, A), dtype=torch.bool, device=dev)
    rew_tb = torch.empty((T, B), dtype=torch.float32, device=dev)
    done_tb = torch.empty((T, B), dtype=torch.bool, device=dev)
    succ_tb = torch.empty((T, B), dtype=torch.bool, device=dev)

    def episode_replay():
        # one launch plays the whole resident action stream (qg_replay); state stays in the SMs between steps
        env.restore()
        env.replay(actions, coins=coins, obs=obs_ring, mask=mask_ring, reward=rew_tb, done=done_tb, success=succ_tb)

    def episode_steps():
        # policy-in-the-loop granularity: one fused launch per env-step (qg_step)
        env.restore()
        for t in range(T):
            env.step(actions[t], coins=None if coins is None else coins[t], obs=obs_ring[t % nbuf], mask=mask_ring[t % nbuf])

    stream = torch.cuda.Stream(device=dev)
    sampler = ClockSampler(local)

    def capture(fn):
        with torch.cuda.stream(stream):
            fn()
            stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                fn()
            stream.synchronize()
        return g

    def timed(graph, sample_clocks=False):
        """W warm-ups, then K replays of the captured episode, CUDA events on the launching stream."""
        with torch.cuda.stream(stream):
            for _ in range(max(Wm, 3)):
                graph.replay()
            stream.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0 = time.time()
            ev0.record(stream)
            for _ in range(K):
                graph.replay()
            ev1.record(stream)
            stream.synchronize()
            w1 = time.time()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t_ms = ev0.elapsed_time(ev1)
        # the sampler has been running since the pre-spin of the same graph (about 1 s of identical load right before
        # the timed replays): the median covers that load window and the timed region
        clk = sampler.stop(load_t0[0], w1) if (sample_clocks and rank == 0) else None
        if world > 1:
            tms = torch.tensor([t_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            t_ms = float(tms.item())
        return t_ms, clk

    g_replay = capture(episode_replay)
    g_steps = None if args.no_per_step else capture(episode_steps)
    # bring the GPU out of its idle power state before anything is timed (the first launches after process start-up
    # otherwise run at idle clocks): about one second of the replay graph
    load_t0 = [time.time()]
    if rank == 0:
        sampler.start()
    with torch.cuda.stream(stream):
        t_end = time.time() + 1.0
        while time.time() < t_end:
            for _ in range(20):
                g_replay.replay()
            stream.synchronize()
    load_t0[0] = time.time() - 0.7               # clock samples of the last 0.7 s of the pre-spin count as "under load"
    ms, clocks = timed(g_replay, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, obs_ring, mask_ring, rew_tb, done_tb, succ_tb)
    ms_steps = timed(g_steps)[0] if g_steps is not None else None
    packed = None
    if not args.no_packed and not (kind == W.PERM and n > 64):
        # the same episode with the observation delivered as packed bits (SURVEY.md §8f row 3): 1 bit per entry instead of an f32,
        # no mask tensor (masks() is [!success; A], the success flag carries it)
        ow = env.obs_words()
        bits_ring = env.new_obs_bits(ring=nbuf)

        def episode_replay_bits():
            env.restore()
            env.replay_bits(actions, obs_bits=bits_ring, coins=coins, reward=rew_tb, done=done_tb, success=succ_tb)

        ms_bits = timed(capture(episode_replay_bits))[0]
        packed = {"value": world * B * T * K / (ms_bits * 1e-3), "unit": UNIT, "ms_per_step": ms_bits / K,
                  "bytes_per_env_step": 4 * ow + 4 + 4 + 1 + 1,
                  "note": "qg_replay_bits: observation as uint32 bit words [B][ceil(obs/32)] for the fused policy kernel (qg_policy_forward_bits); "
                          "outputs per env-step: packed obs + f32 reward + u8 done + u8 success, input int32 action"}
    total_env_steps = world * B * T * K
    value = total_env_steps / (ms * 1e-3)
    errs = int(env.errors().max().item())

    # ---- e2e: the same episode through the host-buffer C-ABI calls ---------------------------------------
    e2e = None
    if not args.no_e2e:
        Ke = max(1, min(K, 10))
        tiles = env.flag_words()

        def host_timed(fn, reps):
            with torch.cuda.stream(stream):
                fn()
                stream.synchronize()
                if world > 1:
                    dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(reps):
                    fn()
                e1.record(stream)
                stream.synchronize()
                t_ms = e0.elapsed_time(e1)
            if world > 1:
                t2 = torch.tensor([t_ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
                t_ms = float(t2.item())
            return t_ms

        e2e_packed = None
        if A <= 256:
            # packed wire format (qg_replay_host_packed): uint8 actions in; f32 reward + 2 bits per env-step of is_final / success out;
            # pinned buffers on the GPU's NUMA node (qg_host_alloc)
            h_a8 = env.host_buffer((T, B), np.uint8); h_a8[:] = actions_h.astype(np.uint8)
            h_rw = env.host_buffer((T, B), np.float32)
            h_db = env.host_buffer((tiles, T), np.uint32); h_sb = env.host_buffer((tiles, T), np.uint32)
            h_c8 = None
            if coins is not None:
                h_c8 = env.host_buffer((T, B), np.uint8); h_c8[:] = coins.cpu().numpy()

            def episode_host_packed():
                env.restore()
                env.replay_host_packed(h_a8, h_db, h_sb, reward=h_rw, coins=h_c8, obs=obs_ring, mask=mask_ring)
                return float(h_rw[T - 1, 0]) + float(h_db[0, T - 1] & 1)

            rew_dev_tb = torch.empty((T, B), dtype=torch.float32, device=dev)

            def episode_host_flags_only():
                # learner on the device: rewards stay in HBM (for a device-side return / qg_gae), only the flags travel
                env.restore()
                env.replay_host_packed(h_a8, h_db, h_sb, reward_dev=rew_dev_tb, coins=h_c8, obs=obs_ring, mask=mask_ring)
                return float(h_db[0, T - 1] & 1)

            # the same call, two episodes in flight (qg_replay_host_packed_async): episode i + 1 is queued (its own reward / flag buffers) before
            # the host waits for episode i and reads its results, so the device does not idle across the host's turn-around
            h_rw2 = [h_rw, env.host_buffer((T, B), np.float32)]
            h_db2 = [h_db, env.host_buffer((tiles, T), np.uint32)]; h_sb2 = [h_sb, env.host_buffer((tiles, T), np.uint32)]

            def submit(i):
                env.restore()
                env.replay_host_packed(h_a8, h_db2[i & 1], h_sb2[i & 1], reward=h_rw2[i & 1], coins=h_c8, obs=obs_ring, mask=mask_ring, sync=False)
                ev = torch.cuda.Event()
                ev.record(stream)
                return ev

            def collect(i):
                return float(h_rw2[i & 1][T - 1, 0]) + float(h_db2[i & 1][0, T - 1] & 1)

            def pipelined(reps):
                with torch.cuda.stream(stream):
                    submit(0).synchronize(); collect(0)
                    stream.synchronize()
                    if world > 1:
                        dist.barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    pending = None
                    for i in range(reps):
                        ev = submit(i)
                        if pending is not None:
                            pending[0].synchronize(); collect(pending[1])
                        pending = (ev, i)
                    pending[0].synchronize(); collect(pending[1])
                    e1.record(stream)
                    stream.synchronize()
                    t_ms = e0.elapsed_time(e1)
                if world > 1:
                    t2 = torch.tensor([t_ms], dtype=torch.float64, device=dev)
                    dist.all_reduce(t2, op=dist.ReduceOp.MAX)
                    t_ms = float(t2.item())
                return t_ms

            sms = host_timed(episode_host_packed, Ke)          # one episode at a time: the call synchronises
            fms = host_timed(episode_host_flags_only, Ke)
            pms = pipelined(Ke)
            e2e_packed = {"value": world * B * T * Ke / (pms * 1e-3), "ms": pms, "sync_value": world * B * T * Ke / (sms * 1e-3),
                          "h2d": T * B * (1 + (1 if h_c8 is not None else 0)), "d2h": T * B * 4 + 2 * tiles * T * 4,
                          "flags_only": world * B * T * Ke / (fms * 1e-3), "numa_node": getattr(env, "numa_node", -1)}

        pin_a = torch.from_numpy(actions_h).pin_memory()
        a_np = pin_a.numpy()
        pin_c = None if coins is None else coins.cpu().pin_memory()
        c_np = None if pin_c is None else pin_c.numpy()
        rew = torch.empty((T, B), dtype=torch.float32).pin_memory(); don = torch.empty((T, B), dtype=torch.uint8).pin_memory(); suc = torch.empty((T, B), dtype=torch.uint8).pin_memory()
        rew_np, don_np, suc_np = rew.numpy(), don.numpy(), suc.numpy()

        def episode_host():
            # the round-1 wire format (qg_replay_host): int32 actions, f32 reward + u8 done + u8 success
            env.restore()
            env.replay_host(a_np, rew_np, don_np, suc_np, coins=c_np, obs=obs_ring, mask=mask_ring)
            return float(rew_np[T - 1, 0])

        def episode_host_per_step():
            # a host-side collector: one synchronous call per env-step (qg_step_host)
            env.restore()
            acc = 0.0
            for t in range(T):
                env.step_host(a_np[t], rew_np[0], don_np[0], suc_np[0], coins=None if c_np is None else c_np[t], obs=obs_ring[t % nbuf], mask=mask_ring[t % nbuf])
                acc += float(rew_np[0, 0])
            return acc

        ems = host_timed(episode_host, Ke)
        Ks = max(1, min(K, 3))
        ems_ps = host_timed(episode_host_per_step, Ks)
        wide = world * B * T * Ke / (ems * 1e-3)
        e2e = {"value": e2e_packed["value"] if e2e_packed else wide, "unit": UNIT,
               "h2d_bytes_per_step": e2e_packed["h2d"] if e2e_packed else T * B * (4 + (1 if c_np is not None else 0)),
               "d2h_bytes_per_step": e2e_packed["d2h"] if e2e_packed else T * B * 6,
               "note": ("qg_replay_host_packed_async, pinned NUMA-local host buffers, two episodes in flight (episode i + 1 is queued, with its own output buffers, "
                        "before the host waits for episode i and reads its rewards / flags): every episode's uint8 actions [T][B] are copied from pinned host memory "
                        "by the copy engine in flagged chunks while the kernel plays; f32 reward [T][B] and the is_final / success bit planes uint32[B/32][T] are "
                        "written by the kernel to host memory and read by the host; one launch per episode, obs + mask stay on the device (it can exceed the device-resident "
                        "`value`, whose launch also writes int32-action-stream-sized reward / done / success tensors to HBM: here those streams leave over PCIe).  sync_value: "
                        "qg_replay_host_packed, one episode at a time (the call returns when the stream is synchronised)") if e2e_packed else "qg_replay_host (int32 actions; f32 reward, u8 done, u8 success)",
               "steps": Ke,
               "sync_value": e2e_packed["sync_value"] if e2e_packed else wide,             # one episode at a time, synchronous call
               "flags_only_value": e2e_packed["flags_only"] if e2e_packed else None,        # rewards kept on the device
               "int32_u8_format_value": wide,                                              # round-1 wire format: 10 B per env-step
               "per_step_sync_value": world * B * T * Ks / (ems_ps * 1e-3),                # qg_step_host: one synchronous call per env-step
               "host_numa_node": e2e_packed["numa_node"] if e2e_packed else -1}

    synth = None if args.no_synth else run_synth(args, dev, local, rank, world)
    collector = None if args.no_collector else run_collector(args, dev, local, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    algo = ALGO_BYTES.get(args.config)
    launch_us = ms * 1e3 / K                       # one replay launch (T env-steps for every env) + the 6 MB restore copy
    step_launch_us = ms_steps * 1e3 / (T * K) if ms_steps else None
    roofline = None
    per_step = None
    if algo:
        st_b = STATE_BYTES.get(args.config, 0)
        launch_bytes = (T * (algo - st_b) + st_b) * B          # record moved once per launch, streams T times
        achieved = launch_bytes / (launch_us * 1e-6) / 1e9
        traffic = TRAFFIC_BYTES_PER_LAUNCH.get((args.config, B, T))
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                    "kernel": f"qg::k_step<{args.config.split('_')[1]},STEP> nsteps={T} (qg_replay)", "algorithmic_bytes_per_env_step": algo,
                    "algorithmic_bytes_per_launch": launch_bytes, "avg_launch_us": launch_us,
                    "note": f"one launch = {T} env-steps for every env: the obs/mask/reward/done/action streams ({algo - st_b} B per env-step) move "
                            f"every env-step, the packed state + metrics record ({st_b} B, read + write) once per launch; "
                            "peak is the measured device-copy bandwidth (a write-only fill reaches 7 426 GB/s on this part, tools/store_ceiling.py)"}
        ach1 = algo * B / (step_launch_us * 1e-6) / 1e9 if ms_steps else None
        per_step = None if not ms_steps else {"value": world * B * T * K / (ms_steps * 1e-3), "unit": UNIT, "avg_launch_us": step_launch_us, "launches": T * K,
                    "roofline_achieved_gbs": ach1, "roofline_frac": ach1 / peak,
                    "note": "one fused launch per env-step (qg_step, policy-in-the-loop granularity), programmatic dependent launch, CUDA graph"}
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:          # the CPU figure is reported beside the 1-GPU run only
        threads = os.cpu_count() or 1
        envs = args.cpu_sample_envs or B                       # the GPU arm's own batch; passes repeated until ~12 s of CPU work
        probe = cpu_run(args, envs, threads=threads)
        passes = max(1, min(40, int(12.0 / max(probe["seconds"], 1e-3))))
        r = cpu_run(args, envs, steps=passes, threads=threads)
        envs1 = max(256, int(probe["value"] / threads * 3.0 / T) // 64 * 64)          # ~3 s on one thread (SURVEY.md §8d: one thread and all threads)
        r1 = cpu_run(args, envs1, threads=1)
        cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"{passes} passes of {envs} envs x {T} env-steps (the GPU arm's batch, targets and action stream distribution), oracle C++ port of the "
                                  f"Rust core, per env-step step+observe+masks+reward+is_final, {threads} host threads, {r['seconds']:.1f} s",
                        "single_thread": {"value": r1["value"], "unit": UNIT, "cores": 1, "sample": f"{envs1} envs x {T} env-steps, {r1['seconds']:.1f} s"}}
    if e2e is not None and synth is not None:
        # (the driver's parser keeps scalar keys of `e2e`: the second BASELINE.json metric rides there as well as in `synth`)
        e2e["synth_weak_rollouts_per_s"] = synth["value"]
        e2e["synth_strong_rollouts_per_s"] = synth["strong"]["value"]
    line = {
        "metric": METRIC if args.config == "C3_clifford8_full" else f"batched env-steps/sec ({args.config})",
        "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 bit-planes (GF(2)) + f32 reward/obs", "data": "synthetic",
        "config": config_json(args, world), "obs_buffers": nbuf, "cuda_graph": True, "tile_envs": args.tile_envs,
        "clocks": clocks, "e2e": e2e, "gpu_launches": K, "roofline": roofline, "per_step_launch": per_step, "cpu_baseline": cpu_baseline,
        "packed_obs": packed, "synth": synth, "collector": collector, "engine_error_flags": errs,
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_collector(args, dev, local, rank, world):
    """Policy-in-the-loop data collection on the bench config (what twisterl's PPO collector does on CPU cores, rl/configs.py:133-137):
    every decision = selective reset + observe + PyTorch BasicPolicy forward + Philox sample + fused step, then GAE on the device.
    Reported as env-steps/s including the policy; the env-only numbers above are its upper bound."""
    import torch
    import torch.distributed as dist
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200 import workloads as W
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.search import BasicPolicy

    kind, n, gateset, kw = workload(args)
    B, T = min(args.envs, 65536), 32
    pk = dict(kw)
    if kind != W.PAULI:
        pk["add_inverts"] = False
    env = BatchedEnv(kind, n, gateset, B, device=local, difficulty=64, depth_slope=2, max_depth=128, add_perms=False, **pk)
    torch.manual_seed(0)
    pol = BasicPolicy(env.obs_shape(), len(gateset), embedding_size=512, common_layers=(256,))
    def leg(precision):
        col = RolloutCollector(env, pol, use_twists=False, seed=rank, matmul_precision=precision)
        col.collect(4)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ro = col.collect(T)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        episodes, _ = ro.episode_stats()
        return {"value": world * B * T / (ms * 1e-3), "unit": UNIT, "ms_per_decision": ms / T, "episodes_finished": episodes}

    def leg_packed():
        col = RolloutCollector(env, pol, use_twists=False, seed=rank)
        col.collect_packed(T)              # eager (lazy initialisation)
        col.collect_packed(T)              # captured into a CUDA graph and replayed
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ro = col.collect_packed(T)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        episodes, _ = ro.episode_stats()
        return {"value": world * B * T / (ms * 1e-3), "unit": UNIT, "ms_per_decision": ms / T, "episodes_finished": episodes}

    out = leg("f32")
    out.update({"envs_per_gpu": B, "decisions": T,
                "note": "RolloutCollector.collect: reset_select + observe (dense f32) + PyTorch BasicPolicy 512/256 forward (f32 cuBLAS) + softmax + "
                        "qg_collect_step + log-prob gather per decision, qg_gae at the end; difficulty 64, random-init policy",
                "tf32_policy": dict(leg("tf32"), note="same collector with matmul_precision='tf32' (the policy's GEMMs on tensor cores, f32 accumulate)"),
                "bf16_policy": dict(leg("bf16"), note="same collector with matmul_precision='bf16' (torch.autocast)")})
    try:
        out["tensor_core_packed"] = dict(leg_packed(), note="RolloutCollector.collect_packed: packed-bit observations + the policy on tcgen05 tensor cores "
                                                           "(qg_policy_tc_forward_bits: f16 hi+lo split operands, f32 accumulate, logits within 1e-4 of the f32 module) + qg_collect_step")
    except Exception as ex:          # (reported, not hidden: the leg is the newest kernel)
        out["tensor_core_packed"] = {"error": repr(ex)[:300]}
    return out


def run_synth(args, dev, local, rank, world):
    """Second BASELINE.json metric: synth rollouts/sec on configs[4] (PermutationGym 27q heavy-hex, `num_searches = 1000`): policy-guided
    rollouts on the device (BasicPolicy-shaped MLP 729->512->256->{28,1}, torch.manual_seed(0) init, sampling), the whole search one launch of
    qg_search_run, the best rollout reduced on the GPU and across ranks by qg_search_finish (one NCCL all-gather + on-GPU pick through the
    C ABI's own communicator).  Two readings of "across 1/2/4/8 GPUs": WEAK = 1000 rollouts per GPU (1000 x N per search), STRONG = ONE
    1000-rollout search split over the N GPUs (1000 / N rollouts each, global rollout ids, the same winner for every N).  Wall time of
    whole solve() calls, max over ranks."""
    import torch
    import torch.distributed as dist
    from qiskit_gym_b200 import engine
    from qiskit_gym_b200 import workloads as W
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch

    kind, n, gateset, kw = W.baseline_configs()["C5_perm27_heavyhex"]
    R = args.synth_rollouts
    rng = np.random.Generator(np.random.PCG64(20261017 + 5))
    targets = [rng.permutation(n).astype(np.int64).tolist() for _ in range(args.synth_searches + 1)]
    shallow = list(range(n)); shallow[0], shallow[1] = shallow[1], shallow[0]      # one SWAP away: exercises the success / early-exit path
    comm = engine.nccl_comm_create(local) if world > 1 else None

    def leg(backend, rollouts, use_comm=True):
        torch.manual_seed(0)
        pol = BasicPolicy([n, n], len(gateset), embedding_size=512, common_layers=(256,))
        rs = RolloutSearch(kind, n, gateset, pol, rollouts, device=local, max_depth=128, add_inverts=False, policy_backend=backend)
        c = comm if use_comm else None
        rs.solve(targets[0], deterministic=False, seed=0, first_rollout_id=rank * rollouts, comm=c)    # warm-up: graph capture, cuBLAS
        res_sh = rs.solve(shallow, deterministic=False, seed=1, first_rollout_id=rank * rollouts, comm=c)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        its = 0
        for i in range(args.synth_searches):
            r = rs.solve(targets[1 + i], deterministic=False, seed=2 + i, first_rollout_id=rank * rollouts, comm=c)
            its += r.iterations
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        total = world * rollouts * args.synth_searches
        return {"value": total / sec, "unit": "rollouts/s", "rollouts_per_gpu": rollouts, "rollouts_per_search": world * rollouts,
                "decisions_per_search": its / max(args.synth_searches, 1),
                "us_per_decision": 1e6 * sec / max(its, 1), "ms_per_search": 1e3 * sec / max(args.synth_searches, 1),
                "shallow_target": {"success": bool(res_sh.success), "circuit_len": None if res_sh.actions is None else len(res_sh.actions),
                                   "key": int(res_sh.key), "decisions": res_sh.iterations, "ms": 1e3 * res_sh.seconds}}

    out = {"metric": "synth rollouts/sec (PermutationGym 27q heavy-hex, num_searches=1000)", "searches": args.synth_searches}
    out.update(leg("persistent", R))
    out["scaling"] = "weak: num_searches = 1000 per GPU"
    out["policy_backend"] = ("persistent: the whole search is ONE launch of qg_search_run (each CTA owns 8 rollouts and loops packed observation -> "
                             "fused policy network -> Philox sample + env step); cross-GPU best by qg_search_finish (NCCL all-gather + on-GPU pick)")
    if R % world == 0:
        out["strong"] = dict(leg("persistent", R // world), scaling=f"strong: ONE num_searches = {R} search split over {world} GPU(s), {R // world} rollouts each",
                             note="latency-bound: a search is <= 128 sequential decisions whatever the number of rollouts per GPU, so splitting one search shortens "
                                  "nothing but the per-decision work; the winner (key, actions) is identical for every GPU count (tools/multi_gpu_parity.py)")
    else:
        out["strong"] = {"value": None, "note": f"{R} rollouts do not split evenly over {world} GPUs"}
    if args.synth_all_backends:
        out["two_kernel"] = dict(leg("fused", R, use_comm=False), note="qg_policy_forward_bits + qg_search_step_bits per decision, CUDA graph, PDL; torch.distributed reduction")
        out["torch_policy"] = dict(leg("torch", R, use_comm=False), note="same search with the PyTorch BasicPolicy on dense f32 observations (cuBLAS GEMMs + softmax + qg_search_step)")
    out["note"] = ("uniform random 27-permutations, random-init policy (no checkpoint exists for this map): rollouts run to max_depth=128; "
                   "time is host wall clock over whole solve() calls (set_state broadcast, one search launch, on-GPU best reduction, "
                   "cross-rank all-gather), max over ranks")
    if comm is not None:
        engine.nccl_comm_destroy(comm)
    return out


JSON_OUT = sys.stdout


def main():
    global JSON_OUT
    args = parse_args()
    # stdout carries exactly one JSON line: keep a private handle on the real stdout for it and point file descriptor 1 at stderr, so
    # that nothing a library prints there (NCCL's version banner, a warning from a C extension) can land beside the line
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
