"""BatchedEnv — B independent synthesis environments stepped by one fused CUDA launch.

Host-side mirror of the reference's raw-env interface (`impl twisterl::rl::env::Env for
{Permutation, LinearFunction, Clifford, PauliEnv}`, e.g. rust/src/envs/clifford.rs:285-382) with a
leading batch dimension.  PyTorch only provides device memory and streams; every computation is a
call into the C ABI (include/qg_engine.h).
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np
import torch

from . import _abi
from ._lib import check, lib


def _dptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class BatchedEnv:
    def __init__(self, env_kind: int, num_qubits: int, gateset: Iterable, batch: int, device: int | None = None,
                 difficulty: int = 1, depth_slope: int = 2, max_depth: int = 128, **kwargs):
        L = lib()
        gateset = list(gateset)
        gates = _abi.parse_gateset(gateset, L.qg_gate_kind_from_name)
        self._gateset = [(str(n), tuple(int(q) for q in idx)) for n, idx in gateset]
        self.cfg = _abi.make_config(env_kind, num_qubits, difficulty, gates, len(self._gateset), depth_slope, max_depth, **kwargs)
        check(L.qg_config_validate(C.byref(self.cfg)))
        if not torch.cuda.is_available():
            raise RuntimeError("qiskit_gym_b200 needs a CUDA device (no CPU fallback)")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.batch = int(batch)
        nbytes = check(L.qg_workspace_bytes(C.byref(self.cfg), self.batch))
        self._workspace = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.device)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(L.qg_create(C.byref(self.cfg), self.device_index, self.batch, _dptr(self._workspace), C.byref(h)))
        self._h = h
        shp = (C.c_int32 * 2)()
        L.qg_obs_shape(self._h, shp)
        self._obs_shape = (int(shp[0]), int(shp[1]))
        self._obs_size = int(L.qg_obs_size(self._h))
        self._A = int(L.qg_num_actions(self._h))
        B = self.batch
        dev = self.device
        self.obs = torch.zeros((B,) + self._obs_shape, dtype=torch.float32, device=dev)
        self.mask = torch.zeros((B, self._A), dtype=torch.bool, device=dev)
        self.reward = torch.zeros(B, dtype=torch.float32, device=dev)
        self.done = torch.zeros(B, dtype=torch.bool, device=dev)
        self.success = torch.zeros(B, dtype=torch.bool, device=dev)
        self._twists = None
        self.search_key = (0, 0)            # (seed, first rollout id) of the last search_begin

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().qg_destroy(h)
                for p in getattr(self, "_host_bufs", []):
                    lib().qg_host_free(p)
            except Exception:
                pass
            self._h = None

    # ------------------------------------------------------------------ shape / config
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def obs_shape(self):
        return list(self._obs_shape)

    def num_actions(self):
        return self._A

    @property
    def gateset(self):
        return list(self._gateset)

    @property
    def difficulty(self):
        return int(lib().qg_get_difficulty(self._h))

    @difficulty.setter
    def difficulty(self, d):
        check(lib().qg_set_difficulty(self._h, int(d)))

    def twists(self):
        """(obs_perms, act_perms) of Env::twists (symmetry.rs:297-361)."""
        if self._twists is None:
            L = lib()
            t = C.c_void_p()
            check(L.qg_twists_create(C.byref(self.cfg), C.byref(t)))
            try:
                cnt, ol, al = L.qg_twists_count(t), L.qg_twists_obs_len(t), L.qg_twists_act_len(t)
                obs = np.zeros((cnt, ol), dtype=np.int64)
                act = np.zeros((cnt, al), dtype=np.int64)
                check(L.qg_twists_copy(t, obs.ctypes.data_as(C.c_void_p), act.ctypes.data_as(C.c_void_p)))
            finally:
                L.qg_twists_destroy(t)
            self._twists = (obs.tolist(), act.tolist())
        return self._twists

    # ------------------------------------------------------------------ state in
    @staticmethod
    def _payload_rows(states) -> np.ndarray:
        """A sequence / int64 array of payloads -> int64 [count, stride], shorter payloads zero-padded."""
        if isinstance(states, np.ndarray) and states.ndim == 2:
            return np.ascontiguousarray(states, dtype=np.int64)
        arr = np.zeros((len(states), max((len(s) for s in states), default=1)), dtype=np.int64)
        for i, s in enumerate(states):
            arr[i, : len(s)] = s
        return arr

    def set_state(self, states, first: int = 0):
        """Env::set_state.  `states`: one payload (list[int]) => loaded into every env, or a sequence /
        int64 array of per-env payloads."""
        if (isinstance(states, np.ndarray) and states.ndim == 2) or (len(states) > 0 and isinstance(states[0], (list, tuple, np.ndarray))):
            arr = self._payload_rows(states)
            count, stride, bcast = arr.shape[0], arr.shape[1], 0
        else:
            arr = np.asarray(list(states), dtype=np.int64).reshape(1, -1)
            count, stride, bcast = self.batch - first, arr.shape[1], 1
        with torch.cuda.device(self.device):
            check(lib().qg_set_state(self._h, arr.ctypes.data_as(C.c_void_p), stride, first, count, bcast, self._stream()))

    def set_state_grouped(self, states, group: int):
        """Env::set_state for groups of envs (qg_set_state_grouped): payload p of `states` (a sequence / int64 array of payloads) goes
        to envs [p * group, (p + 1) * group); envs past len(states) * group are untouched."""
        arr = self._payload_rows(states)
        with torch.cuda.device(self.device):
            check(lib().qg_set_state_grouped(self._h, arr.ctypes.data_as(C.c_void_p), arr.shape[1], arr.shape[0], int(group), self._stream()))

    def reset(self, seed: int = 0, first_env_id: int = 0):
        check(lib().qg_reset(self._h, C.c_uint64(seed & (2**64 - 1)), first_env_id, self._stream()))

    def reset_select_dev(self, seed_dev: torch.Tensor, first_env_id: int = 0, select: torch.Tensor | None = None):
        """reset_select with the seed read from device memory at run time (int64 tensor, 1 element): CUDA-graph replays."""
        assert seed_dev.is_cuda and seed_dev.element_size() == 8
        check(lib().qg_reset_select_dev(self._h, _dptr(seed_dev), first_env_id, _dptr(select), self._stream()))

    def collect_step_dev(self, weights: torch.Tensor, seed_dev: torch.Tensor, deterministic: bool = False, chosen: torch.Tensor | None = None,
                         reward: torch.Tensor | None = None, done: torch.Tensor | None = None, success: torch.Tensor | None = None):
        """collect_step with the seed read from device memory at run time; no observation / mask output."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous() and seed_dev.is_cuda and seed_dev.element_size() == 8
        check(lib().qg_collect_step_dev(self._h, _dptr(seed_dev), _dptr(weights), 1 if deterministic else 0, None, None, _dptr(chosen),
                                        _dptr(self.reward if reward is None else reward), _dptr(self.done if done is None else done),
                                        _dptr(self.success if success is None else success), self._stream()))

    def collect_step_twisted_dev(self, weights: torch.Tensor, act_table: torch.Tensor, twist: torch.Tensor, seed_dev: torch.Tensor,
                                 deterministic: bool = False, chosen: torch.Tensor | None = None, policy_chosen: torch.Tensor | None = None,
                                 reward: torch.Tensor | None = None, done: torch.Tensor | None = None, success: torch.Tensor | None = None):
        """collect_step_dev for a twisted collector (qg_collect_step_twisted_dev): `weights` [B, A] are in the policy's twisted action order,
        env action g of env i takes weights[i, act_table[twist[i], g]]; `policy_chosen` receives act_table[twist[i], chosen] (-1: not stepped)."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous() and seed_dev.is_cuda and seed_dev.element_size() == 8
        assert act_table.dtype == torch.int32 and act_table.is_contiguous() and act_table.shape[1] == self._A
        assert twist.dtype == torch.int32 and twist.is_contiguous() and twist.numel() == self.batch
        assert policy_chosen is None or (policy_chosen.dtype == torch.int32 and policy_chosen.numel() == self.batch)
        check(lib().qg_collect_step_twisted_dev(self._h, _dptr(seed_dev), _dptr(weights), _dptr(act_table), _dptr(twist), 1 if deterministic else 0,
                                                _dptr(chosen), _dptr(policy_chosen), _dptr(self.reward if reward is None else reward),
                                                _dptr(self.done if done is None else done), _dptr(self.success if success is None else success),
                                                self._stream()))

    def reset_select(self, seed: int = 0, first_env_id: int = 0, select: torch.Tensor | None = None):
        """Env::reset for the envs flagged in `select` (bool/uint8 [B]) or, with select=None, for every env that is final."""
        assert select is None or (select.is_cuda and select.numel() == self.batch and select.element_size() == 1)
        check(lib().qg_reset_select(self._h, C.c_uint64(seed & (2**64 - 1)), first_env_id, _dptr(select), self._stream()))

    def snapshot(self):
        """Clone of the whole batch (device copy of every env record)."""
        check(lib().qg_snapshot(self._h, self._stream()))

    def restore(self):
        check(lib().qg_restore(self._h, self._stream()))

    # ------------------------------------------------------------------ fused step
    def step(self, actions: torch.Tensor, coins: torch.Tensor | None = None, perm_raw: torch.Tensor | None = None,
             obs: torch.Tensor | None | bool = True, mask: torch.Tensor | None | bool = True):
        """One fused step for all envs.  `actions`: int32 CUDA tensor [B].  obs/mask: True = write into the
        engine-owned tensors, None/False = skip, or a caller tensor to write into.  Returns (obs, reward, done)."""
        assert actions.dtype == torch.int32 and actions.is_cuda and actions.numel() == self.batch
        obs_t = self.obs if obs is True else (None if obs is False else obs)
        mask_t = self.mask if mask is True else (None if mask is False else mask)
        check(lib().qg_step(self._h, _dptr(actions), _dptr(coins), _dptr(perm_raw), _dptr(obs_t), _dptr(mask_t),
                            _dptr(self.reward), _dptr(self.done), _dptr(self.success), self._stream()))
        return obs_t, self.reward, self.done

    def replay(self, actions: torch.Tensor, coins: torch.Tensor | None = None, perm_raw: torch.Tensor | None = None,
               obs: torch.Tensor | None = None, mask: torch.Tensor | None = None, reward: torch.Tensor | None = None,
               done: torch.Tensor | None = None, success: torch.Tensor | None = None):
        """T consecutive fused steps in one launch from a resident action stream `actions` int32[T, B] (qg_replay).
        obs: float32[ring, B, obs...] / mask: bool[ring, B, A] ring buffers (step t writes slot t % ring; both must have the
        same ring), reward float32[T, B], done / success bool[T, B]; any of them may be None."""
        assert actions.dtype == torch.int32 and actions.is_cuda and actions.is_contiguous() and actions.shape[-1] == self.batch
        T = int(actions.shape[0]) if actions.dim() == 2 else 1
        ring = 1
        if obs is not None:
            assert obs.is_contiguous() and obs.numel() % (self.batch * self._obs_size) == 0
            ring = obs.numel() // (self.batch * self._obs_size)
        if mask is not None:
            assert mask.is_contiguous() and mask.numel() % (self.batch * self._A) == 0
            mring = mask.numel() // (self.batch * self._A)
            assert obs is None or mring == ring, "obs and mask rings differ"
            ring = mring
        for t in (coins, perm_raw, reward, done, success):
            assert t is None or (t.is_contiguous() and t.numel() == T * self.batch)
        check(lib().qg_replay(self._h, T, _dptr(actions), _dptr(coins), _dptr(perm_raw), _dptr(obs), _dptr(mask), ring,
                              _dptr(reward), _dptr(done), _dptr(success), self._stream()))

    def replay_host(self, actions: np.ndarray, reward: np.ndarray | None = None, done: np.ndarray | None = None,
                    success: np.ndarray | None = None, coins: np.ndarray | None = None, obs: torch.Tensor | None = None,
                    mask: torch.Tensor | None = None):
        """End-to-end episode replay with host buffers (qg_replay_host): int32 actions [T, B] up, reward f32 / done u8 /
        success u8 [T, B] back, chunks pipelined over copy-in / compute / copy-out streams."""
        assert actions.dtype == np.int32 and actions.flags.c_contiguous and actions.shape[-1] == self.batch
        T = int(actions.shape[0])
        ring = 1
        if obs is not None:
            ring = obs.numel() // (self.batch * self._obs_size)
        if mask is not None:
            mring = mask.numel() // (self.batch * self._A)
            assert obs is None or mring == ring, "obs and mask rings differ"
            ring = mring
        for a_, dt in ((reward, np.float32), (done, np.uint8), (success, np.uint8), (coins, np.uint8)):
            assert a_ is None or (a_.dtype == dt and a_.flags.c_contiguous and a_.size == T * self.batch)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        check(lib().qg_replay_host(self._h, T, p(actions), p(coins), _dptr(obs), _dptr(mask), ring, p(reward), p(done), p(success), self._stream()))

    def step_host(self, actions: np.ndarray, reward: np.ndarray, done: np.ndarray, success: np.ndarray | None = None,
                  coins: np.ndarray | None = None, obs: torch.Tensor | None = None, mask: torch.Tensor | None = None):
        """End-to-end step with host buffers (pinned numpy views recommended): H2D actions, fused step
        (observation written to the device tensor `obs`), D2H reward/done/success, stream synchronised."""
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        check(lib().qg_step_host(self._h, p(actions), p(coins), _dptr(obs), _dptr(mask), p(reward), p(done), p(success), self._stream()))

    # ------------------------------------------------------------------ reads
    def observe(self, perm_raw: torch.Tensor | None = None, out: torch.Tensor | None = None):
        out = self.obs if out is None else out
        check(lib().qg_observe(self._h, _dptr(perm_raw), _dptr(out), self._stream()))
        return out

    def masks(self, out: torch.Tensor | None = None):
        out = self.mask if out is None else out
        check(lib().qg_masks(self._h, _dptr(out), self._stream()))
        return out

    def status(self):
        """(reward f32[B], is_final bool[B], success bool[B], depth int32[B]) read back from the records."""
        depth = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
        check(lib().qg_read_status(self._h, _dptr(self.reward), _dptr(self.done), _dptr(self.success), _dptr(depth), self._stream()))
        return self.reward, self.done, self.success, depth

    def metrics(self):
        """uint32[B,4]: n_cnots, n_layers_cnots, n_layers, n_gates (MetricsCounts, metrics.rs:126-133)."""
        out = torch.zeros((self.batch, 4), dtype=torch.int32, device=self.device)
        check(lib().qg_read_metrics(self._h, _dptr(out), self._stream()))
        return out

    def errors(self):
        out = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
        check(lib().qg_read_errors(self._h, _dptr(out), self._stream()))
        return out

    def get_state(self, env: int = 0) -> np.ndarray:
        cap = 1 << 16
        buf = np.zeros(cap, dtype=np.uint8)
        n = C.c_int64()
        check(lib().qg_get_state_host(self._h, env, buf.ctypes.data_as(C.c_void_p), cap, C.byref(n), self._stream()))
        return buf[: n.value].copy()

    def solution(self, env: int = 0) -> list[int]:
        cap = 65536
        buf = np.zeros(cap, dtype=np.uint32)
        n = C.c_int32()
        check(lib().qg_solution_host(self._h, env, buf.ctypes.data_as(C.c_void_p), cap, C.byref(n), self._stream()))
        return [int(v) for v in buf[: n.value]]

    def solutions(self, first: int = 0, count: int | None = None, cap: int | None = None):
        """Env::solution of envs first .. first+count-1 in one kernel + one copy (qg_solutions_host): a list of action lists."""
        count = self.batch - first if count is None else int(count)
        if cap is None:
            cap = max(int(self.cfg.solution_capacity) or (int(self.cfg.max_depth) + 16), 1)
        out = np.zeros((max(count, 1), cap), dtype=np.uint32)
        lens = np.zeros(max(count, 1), dtype=np.int32)
        check(lib().qg_solutions_host(self._h, first, count, out.ctypes.data_as(C.c_void_p), cap, lens.ctypes.data_as(C.c_void_p), self._stream()))
        if (lens[:count] < 0).any():
            raise ValueError(f"a solution is longer than cap={cap}")
        return [out[i, : lens[i]].astype(np.int64).tolist() for i in range(count)]

    # ------------------------------------------------------------------ packed host wire format / NUMA-local pinned memory
    def host_buffer(self, shape, dtype) -> np.ndarray:
        """A pinned host array on the GPU's NUMA node (qg_host_alloc), freed with the engine object."""
        dt = np.dtype(dtype)
        n = int(np.prod(shape))
        p, node = C.c_void_p(), C.c_int32()
        check(lib().qg_host_alloc(self.device_index, n * dt.itemsize, C.byref(p), C.byref(node)))
        self._host_bufs = getattr(self, "_host_bufs", [])
        self._host_bufs.append(p)
        self.numa_node = int(node.value)
        buf = (C.c_uint8 * max(n * dt.itemsize, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)

    def flag_words(self) -> int:
        """Tiles of 32 envs: rows of the packed done / success bit planes uint32[flag_words, T]."""
        return (self.batch + 31) // 32

    def replay_host_packed(self, actions8: np.ndarray, done_bits: np.ndarray, success_bits: np.ndarray | None = None, reward: np.ndarray | None = None,
                           reward_dev: torch.Tensor | None = None, coins: np.ndarray | None = None, obs: torch.Tensor | None = None,
                           mask: torch.Tensor | None = None, sync: bool = True):
        """qg_replay_host_packed: uint8 actions [T, B] in; f32 reward [T, B] (host, or kept on the device in reward_dev) and the
        is_final / success bit planes uint32[ceil(B/32), T] out; pinned buffers (host_buffer) only.  sync=False (qg_replay_host_packed_async):
        returns once the episode is queued on the current stream; the buffers belong to the call until that stream has been waited for."""
        assert actions8.dtype == np.uint8 and actions8.flags.c_contiguous and actions8.shape[-1] == self.batch
        T = int(actions8.shape[0])
        ring = 1
        if obs is not None:
            ring = obs.numel() // (self.batch * self._obs_size)
        if mask is not None:
            mring = mask.numel() // (self.batch * self._A)
            assert obs is None or mring == ring, "obs and mask rings differ"
            ring = mring
        for a_ in (done_bits, success_bits):
            assert a_ is None or (a_.dtype == np.uint32 and a_.flags.c_contiguous and a_.size == self.flag_words() * T)
        assert reward is None or (reward.dtype == np.float32 and reward.flags.c_contiguous and reward.size == T * self.batch)
        assert reward_dev is None or (reward_dev.dtype == torch.float32 and reward_dev.is_contiguous() and reward_dev.numel() == T * self.batch)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        fn = lib().qg_replay_host_packed if sync else lib().qg_replay_host_packed_async
        check(fn(self._h, T, p(actions8), p(coins), _dptr(obs), _dptr(mask), ring, p(reward), _dptr(reward_dev), p(done_bits), p(success_bits), self._stream()))

    def replay_packed(self, actions8: torch.Tensor, done_bits: torch.Tensor | None = None, success_bits: torch.Tensor | None = None,
                      reward: torch.Tensor | None = None, coins: torch.Tensor | None = None, obs: torch.Tensor | None = None, mask: torch.Tensor | None = None):
        """Device-resident form of the packed formats (qg_replay_packed)."""
        assert actions8.dtype == torch.uint8 and actions8.is_cuda and actions8.is_contiguous() and actions8.shape[-1] == self.batch
        T = int(actions8.shape[0])
        ring = 1
        if obs is not None:
            ring = obs.numel() // (self.batch * self._obs_size)
        if mask is not None:
            ring = mask.numel() // (self.batch * self._A)
        check(lib().qg_replay_packed(self._h, T, _dptr(actions8), _dptr(coins), _dptr(obs), _dptr(mask), ring, _dptr(reward),
                                     _dptr(done_bits), _dptr(success_bits), self._stream()))

    @staticmethod
    def unpack_flag_bits(bits: np.ndarray, batch: int) -> np.ndarray:
        """uint32[ceil(B/32), T] bit plane -> uint8[T, B]."""
        tiles, T = bits.shape
        b = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).astype(np.uint8)      # [tile, T, 32]
        return np.ascontiguousarray(b.transpose(1, 0, 2).reshape(T, tiles * 32)[:, :batch])

    # ------------------------------------------------------------------ DLPack
    def dlpack_obs(self, ring: int = 1) -> torch.Tensor:
        """The engine-owned observation ring as a torch tensor through a DLPack capsule (qg_dlpack_obs): zero-copy, float32
        [B, rows, cols] (or [ring, B, rows, cols]); pass it as `obs=` to step / replay.  Must not outlive this object."""
        import ctypes
        m, ptr = C.c_void_p(), C.c_void_p()
        check(lib().qg_dlpack_obs(self._h, int(ring), C.byref(m), C.byref(ptr)))
        new_capsule = ctypes.pythonapi.PyCapsule_New
        new_capsule.restype = ctypes.py_object
        new_capsule.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p]
        cap = new_capsule(m.value, b"dltensor", None)
        t = torch.utils.dlpack.from_dlpack(cap)
        assert t.data_ptr() == ptr.value
        return t

    # ------------------------------------------------------------------ synth search pieces
    def search_finish(self, comm=None, cap: int | None = None):
        """End of a (sharded) search: (key, success, global rollout id, owner rank, actions or None) — qg_search_finish.  `comm`: an
        ncclComm_t handle (nccl_comm_create) or None."""
        if cap is None:
            cap = max(int(self.cfg.solution_capacity) or (int(self.cfg.max_depth) + 16), 1)
        key, ok, rid, owner, n = C.c_int64(), C.c_int32(), C.c_int64(), C.c_int32(), C.c_int32()
        buf = np.zeros(cap, dtype=np.uint32)
        check(lib().qg_search_finish(self._h, comm, C.byref(key), C.byref(ok), C.byref(rid), C.byref(owner), buf.ctypes.data_as(C.c_void_p), cap,
                                     C.byref(n), self._stream()))
        return key.value, bool(ok.value), rid.value, owner.value, ([int(v) for v in buf[: n.value]] if ok.value else None)

    def search_begin(self, seed: int = 0, first_rollout_id: int = 0):
        check(lib().qg_search_begin(self._h, C.c_uint64(seed & (2**64 - 1)), first_rollout_id, self._stream()))
        self.search_key = (seed & (2**64 - 1), int(first_rollout_id))      # (the twisted tree search hands them to its kernels)

    def search_step(self, weights: torch.Tensor, deterministic: bool = False, obs: torch.Tensor | None | bool = True,
                    chosen: torch.Tensor | None = None, num_active: torch.Tensor | None = None):
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous()
        obs_t = self.obs if obs is True else (None if obs is False else obs)
        check(lib().qg_search_step(self._h, _dptr(weights), 1 if deterministic else 0, _dptr(obs_t), None, _dptr(chosen),
                                   _dptr(num_active), self._stream()))
        return obs_t

    def collect_step(self, weights: torch.Tensor, seed: int, deterministic: bool = False, obs: torch.Tensor | None | bool = True,
                     mask: torch.Tensor | None | bool = None, chosen: torch.Tensor | None = None, reward: torch.Tensor | None = None,
                     done: torch.Tensor | None = None, success: torch.Tensor | None = None):
        """Collector decision step (qg_collect_step): sample / arg-max from the action weights, fused env step, and the step's
        reward / is_final / success written per env (untouched for envs that were already final: chosen = -1)."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous()
        obs_t = self.obs if obs is True else (None if obs is False else obs)
        mask_t = self.mask if mask is True else (None if mask is False else mask)
        check(lib().qg_collect_step(self._h, C.c_uint64(seed & (2**64 - 1)), _dptr(weights), 1 if deterministic else 0, _dptr(obs_t), _dptr(mask_t),
                                    _dptr(chosen), _dptr(self.reward if reward is None else reward), _dptr(self.done if done is None else done),
                                    _dptr(self.success if success is None else success), self._stream()))
        return obs_t

    # ------------------------------------------------------------------ packed-bit observations
    def obs_words(self) -> int:
        return int(lib().qg_obs_words(self._h))

    def new_obs_bits(self, ring: int | None = None) -> torch.Tensor:
        shape = (self.batch, self.obs_words()) if ring is None else (ring, self.batch, self.obs_words())
        return torch.zeros(shape, dtype=torch.int32, device=self.device)

    def observe_bits(self, out: torch.Tensor, perm_raw: torch.Tensor | None = None):
        """Env::observe as packed bits: int32 [B, obs_words], bit i%32 of word i//32 = entry i of the flattened observation."""
        assert out.is_cuda and out.element_size() == 4 and out.numel() == self.batch * self.obs_words() and out.is_contiguous()
        check(lib().qg_observe_bits(self._h, _dptr(perm_raw), _dptr(out), self._stream()))
        return out

    def step_bits(self, actions: torch.Tensor, obs_bits: torch.Tensor | None, coins: torch.Tensor | None = None,
                  perm_raw: torch.Tensor | None = None, mask: torch.Tensor | None | bool = None):
        assert actions.dtype == torch.int32 and actions.is_cuda and actions.numel() == self.batch
        mask_t = self.mask if mask is True else (None if mask is False else mask)
        check(lib().qg_step_bits(self._h, _dptr(actions), _dptr(coins), _dptr(perm_raw), _dptr(obs_bits), _dptr(mask_t),
                                 _dptr(self.reward), _dptr(self.done), _dptr(self.success), self._stream()))
        return obs_bits, self.reward, self.done

    def replay_bits(self, actions: torch.Tensor, obs_bits: torch.Tensor | None = None, mask: torch.Tensor | None = None,
                    coins: torch.Tensor | None = None, perm_raw: torch.Tensor | None = None, reward: torch.Tensor | None = None,
                    done: torch.Tensor | None = None, success: torch.Tensor | None = None):
        """qg_replay with packed observations: obs_bits int32 [ring, B, obs_words]."""
        assert actions.dtype == torch.int32 and actions.is_cuda and actions.is_contiguous() and actions.shape[-1] == self.batch
        T = int(actions.shape[0]) if actions.dim() == 2 else 1
        ring = 1
        if obs_bits is not None:
            ring = obs_bits.numel() // (self.batch * self.obs_words())
        if mask is not None:
            mring = mask.numel() // (self.batch * self._A)
            assert obs_bits is None or mring == ring, "obs and mask rings differ"
            ring = mring
        check(lib().qg_replay_bits(self._h, T, _dptr(actions), _dptr(coins), _dptr(perm_raw), _dptr(obs_bits), _dptr(mask), ring,
                                   _dptr(reward), _dptr(done), _dptr(success), self._stream()))

    def search_step_bits(self, weights: torch.Tensor, obs_bits: torch.Tensor | None, deterministic: bool = False,
                         chosen: torch.Tensor | None = None, num_active: torch.Tensor | None = None):
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous()
        check(lib().qg_search_step_bits(self._h, _dptr(weights), 1 if deterministic else 0, _dptr(obs_bits), _dptr(chosen),
                                        _dptr(num_active), self._stream()))
        return obs_bits

    # ------------------------------------------------------------------ record slots (tree search)
    def step_slots(self, src_slot: torch.Tensor, dst_slot: torch.Tensor, actions: torch.Tensor, obs: torch.Tensor | None = None,
                   obs_bits: torch.Tensor | None = None, reward: torch.Tensor | None = None, done: torch.Tensor | None = None,
                   success: torch.Tensor | None = None):
        """Clone + step through record slots (qg_step_slots): logical env i reads slot src_slot[i], plays actions[i] (negative =
        skip) and writes slot dst_slot[i]; outputs are indexed by i.  The engine's batch is the slot pool."""
        count = int(actions.numel())
        for t in (src_slot, dst_slot, actions):
            assert t.dtype == torch.int32 and t.is_cuda and t.is_contiguous() and t.numel() == count
        check(lib().qg_step_slots(self._h, count, _dptr(src_slot), _dptr(dst_slot), _dptr(actions), _dptr(obs), _dptr(obs_bits), None,
                                  _dptr(reward), _dptr(done), _dptr(success), self._stream()))

    def copy_records_from(self, src: "BatchedEnv", dst_slot: torch.Tensor | None = None, count: int | None = None):
        """Copies the records of envs 0..count-1 of `src` into this engine's slots dst_slot[i] (qg_copy_records)."""
        count = src.batch if count is None else int(count)
        assert dst_slot is None or (dst_slot.dtype == torch.int32 and dst_slot.is_cuda and dst_slot.numel() >= count)
        check(lib().qg_copy_records(self._h, _dptr(dst_slot), src._h, count, self._stream()))

    def search_run(self, policy, obs_bits: torch.Tensor, weights: torch.Tensor, max_decisions: int, deterministic: bool = False,
                   decisions: torch.Tensor | None = None):
        """The whole rollout search in one launch (qg_search_run); `policy` is a policy.FusedPolicy.  Call set_state,
        search_begin and observe_bits(obs_bits) first."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous() and weights.numel() == self.batch * self._A
        assert obs_bits.is_cuda and obs_bits.element_size() == 4 and obs_bits.is_contiguous() and obs_bits.numel() == self.batch * self.obs_words()
        assert decisions is None or (decisions.dtype == torch.int32 and decisions.numel() >= (self.batch + 7) // 8)
        check(lib().qg_search_run(self._h, policy._h, 1 if deterministic else 0, int(max_decisions), _dptr(obs_bits), _dptr(weights),
                                  _dptr(decisions), self._stream()))

    # ------------------------------------------------------------------ twisted search (the policy in a symmetry frame per rollout and decision)
    def _twist_args(self, qperm_inv: torch.Tensor, twist: torch.Tensor, act_table: torch.Tensor | None = None):
        assert qperm_inv.dtype == torch.uint8 and qperm_inv.is_cuda and qperm_inv.is_contiguous() and qperm_inv.dim() == 2
        assert qperm_inv.shape[1] == int(self.cfg.num_qubits)
        assert twist.dtype == torch.int32 and twist.is_cuda and twist.is_contiguous() and twist.numel() == self.batch
        assert act_table is None or (act_table.dtype == torch.int32 and act_table.is_cuda and act_table.is_contiguous()
                                     and tuple(act_table.shape) == (qperm_inv.shape[0], self._A))
        return int(qperm_inv.shape[0])

    def search_observe_twisted(self, obs_bits: torch.Tensor, qperm_inv: torch.Tensor, twist: torch.Tensor):
        """qg_search_observe_twisted: after set_state and search_begin, every rollout's packed observation in the frame of its next decision
        (drawn from the engine's seed, the rollout's global id and its step counter) -> obs_bits int32 [B, obs_words], the frames -> twist
        int32 [B].  qperm_inv: uint8 [K, n] (collector.qubit_twist_table)."""
        assert obs_bits.is_cuda and obs_bits.element_size() == 4 and obs_bits.is_contiguous() and obs_bits.numel() == self.batch * self.obs_words()
        K = self._twist_args(qperm_inv, twist)
        check(lib().qg_search_observe_twisted(self._h, _dptr(obs_bits), _dptr(qperm_inv), K, _dptr(twist), self._stream()))
        return obs_bits

    def search_step_twisted(self, weights: torch.Tensor, obs_bits: torch.Tensor, qperm_inv: torch.Tensor, act_table: torch.Tensor,
                            twist: torch.Tensor, deterministic: bool = False, chosen: torch.Tensor | None = None,
                            num_active: torch.Tensor | None = None):
        """search_step_bits of the twisted search (qg_search_step_twisted): env action g of rollout i weighs weights[i, act_table[twist[i], g]];
        the next observation is written in the frame drawn from the post-step counter, twist updated.  act_table: int32 [K, A]."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous() and weights.numel() == self.batch * self._A
        assert obs_bits.is_cuda and obs_bits.element_size() == 4 and obs_bits.is_contiguous() and obs_bits.numel() == self.batch * self.obs_words()
        K = self._twist_args(qperm_inv, twist, act_table)
        check(lib().qg_search_step_twisted(self._h, _dptr(weights), 1 if deterministic else 0, _dptr(obs_bits), _dptr(qperm_inv), _dptr(act_table), K,
                                           _dptr(twist), _dptr(chosen), _dptr(num_active), self._stream()))
        return obs_bits

    def search_run_twisted(self, policy, obs_bits: torch.Tensor, weights: torch.Tensor, max_decisions: int, qperm_inv: torch.Tensor,
                           act_table: torch.Tensor, twist: torch.Tensor, deterministic: bool = False, decisions: torch.Tensor | None = None):
        """search_run of the twisted search (qg_search_run_twisted); call set_state, search_begin and search_observe_twisted(obs_bits, ..,
        twist) first."""
        assert weights.dtype == torch.float32 and weights.is_cuda and weights.is_contiguous() and weights.numel() == self.batch * self._A
        assert obs_bits.is_cuda and obs_bits.element_size() == 4 and obs_bits.is_contiguous() and obs_bits.numel() == self.batch * self.obs_words()
        assert decisions is None or (decisions.dtype == torch.int32 and decisions.numel() >= (self.batch + 7) // 8)
        K = self._twist_args(qperm_inv, twist, act_table)
        check(lib().qg_search_run_twisted(self._h, policy._h, 1 if deterministic else 0, int(max_decisions), _dptr(obs_bits), _dptr(weights),
                                          _dptr(decisions), _dptr(qperm_inv), _dptr(act_table), K, _dptr(twist), self._stream()))

    def search_best(self):
        key, env = C.c_int64(), C.c_int64()
        check(lib().qg_search_best(self._h, C.byref(key), C.byref(env), self._stream()))
        return key.value, env.value

    def search_best_grouped(self, group: int, num_groups: int, cap: int | None = None, out: torch.Tensor | None = None):
        """Best rollout of each group of `group` consecutive envs (qg_search_best_grouped), on the device and without a host
        synchronisation: (keys int64 [num_groups], lens int32 [num_groups], actions int32 [num_groups, cap]); lens[g] = 0 when no rollout
        of group g succeeded, -(length) when its solution is longer than cap.  `out`: an 8-byte aligned int32 device tensor of at least
        num_groups * (3 + cap) elements that the three are views of (so that one copy brings all of them to the host)."""
        if cap is None:
            cap = max(int(self.cfg.solution_capacity) or (int(self.cfg.max_depth) + 16), 1)
        G, need = int(num_groups), int(num_groups) * (3 + int(cap))
        flat = torch.empty(max(need, 2), dtype=torch.int32, device=self.device) if out is None else out
        assert flat.dtype == torch.int32 and flat.is_cuda and flat.is_contiguous() and flat.numel() >= need and flat.data_ptr() % 8 == 0
        keys, lens, actions = flat[: 2 * G].view(torch.int64), flat[2 * G: 3 * G], flat[3 * G: need].view(G, int(cap))
        check(lib().qg_search_best_grouped(self._h, int(group), G, _dptr(keys), _dptr(actions), int(cap), _dptr(lens), self._stream()))
        return keys, lens, actions

    def returns(self):
        out = torch.zeros(self.batch, dtype=torch.float32, device=self.device)
        check(lib().qg_read_returns(self._h, _dptr(out), self._stream()))
        return out


def nccl_comm_create(device: int, group=None):
    """An ncclComm_t of the C ABI's own (qg_nccl_comm_create) over the ranks of a torch.distributed group: rank 0 draws the unique id
    and torch.distributed ships the 128 bytes (any channel would do: a Rust host would use its own)."""
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    idb = (C.c_uint8 * 128)()
    if rank == 0:
        check(lib().qg_nccl_unique_id(idb))
    t = torch.tensor(list(idb), dtype=torch.uint8)
    if dist.get_backend(group) == "nccl":
        t = t.cuda(device)
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    idb = (C.c_uint8 * 128)(*[int(v) for v in t.cpu().tolist()])
    comm = C.c_void_p()
    check(lib().qg_nccl_comm_create(idb, rank, world, int(device), C.byref(comm)))
    return comm


def nccl_comm_destroy(comm):
    check(lib().qg_nccl_comm_destroy(comm))
