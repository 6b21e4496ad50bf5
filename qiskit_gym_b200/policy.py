"""FusedPolicy — the action network of a twisterl `BasicPolicy` evaluated from packed-bit observations by one CUDA kernel
(`qg_policy_forward_bits`, csrc/qg_policy.cu; SURVEY.md §8f row 3).

twisterl's policy consumes `Env::observe()`'s sparse indices with a gather-sum first layer; the PyTorch `BasicPolicy` in
search.py consumes the dense f32 tensor instead.  `FusedPolicy` takes the weights of such a module (or of a checkpoint in
the reference's `.pt` format) and evaluates  obs bits -> Linear -> ReLU -> ... -> Linear -> softmax  in a single launch,
which is what makes a synth-search decision two launches long.  Its output matches the PyTorch module to f32 rounding
(sums run in a different order than cuBLAS'); tests/test_policy.py states the tolerance.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from ._lib import check, lib
from .engine import _dptr


def action_layers(policy: torch.nn.Module):
    """The Linear layers on the observation -> action-logits path of a BasicPolicy-shaped module, in order."""
    layers = [policy.embeddings]
    layers += [m for m in policy.common if isinstance(m, torch.nn.Linear)]
    layers += [m for m in policy.action if isinstance(m, torch.nn.Linear)]
    return layers


def simple_value_head(policy: torch.nn.Module):
    """The value head as (weight [in], bias) when it is a single Linear fed by the same activations as a single-Linear action head (the
    reference's default BasicPolicy and all of its example checkpoints: policy_layers = value_layers = []), else None."""
    act = [m for m in policy.action if isinstance(m, torch.nn.Linear)]
    val = [m for m in getattr(policy, "value", []) if isinstance(m, torch.nn.Linear)]
    if len(act) == 1 and len(val) == 1 and val[0].out_features == 1 and val[0].in_features == act[0].in_features:
        return val[0]
    return None


def weights_version(policy: torch.nn.Module) -> int:
    """Changes whenever a parameter of the module is updated in place (optimizer steps, load_state_dict).  It walks the module tree itself:
    refresh() runs it before every search, and Module.parameters() costs several times as much."""
    v = 0
    for p in policy._parameters.values():
        if p is not None:
            v += p._version
    for m in policy._modules.values():
        if m is not None:
            v += weights_version(m)
    return v


def _host_f32(t: torch.Tensor) -> np.ndarray:
    return np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)


class _PolicyHandle:
    """What FusedPolicy and TensorCorePolicy share: a C handle created from host copies of a BasicPolicy-shaped module's weights (action
    layers, and the value head with with_value), evaluated on packed observation bits, and kept current by refresh().  Subclasses name
    their C entry points (same signatures): _new_handle creates, _forward_fn evaluates, _destroy_fn frees."""

    _forward_fn = _destroy_fn = ""

    def __init__(self, policy: torch.nn.Module, device, with_value: bool):
        if not torch.cuda.is_available():
            raise RuntimeError("qiskit_gym_b200 needs a CUDA device (no CPU fallback)")
        self.device_index = torch.cuda.current_device() if device is None else (device.index if isinstance(device, torch.device) else int(device))
        self.device = torch.device("cuda", self.device_index)
        self.has_value = bool(with_value)
        self._create(policy)

    def _create(self, policy: torch.nn.Module):
        """(Re)creates the C handle from the module's current weights; the previous handle, if any, is destroyed."""
        layers = action_layers(policy)
        ws, bs = [_host_f32(l.weight) for l in layers], [_host_f32(l.bias) for l in layers]
        for a, b in zip(ws[:-1], ws[1:]):
            assert b.shape[1] == a.shape[0], "layers do not chain"
        vw, vb = None, 0.0
        if self.has_value:
            head = simple_value_head(policy)
            if head is None:
                raise NotImplementedError(f"{type(self).__name__}(with_value=True) needs single-Linear action and value heads on the same activations")
            vwa = _host_f32(head.weight).reshape(-1)
            vw, vb = vwa.ctypes.data_as(C.c_void_p), float(head.bias.detach().cpu().numpy().reshape(-1)[0])
        n = len(ws)
        out_features = [int(w.shape[0]) for w in ws]
        h = self._new_handle(int(ws[0].shape[1]), n, (C.c_int32 * n)(*out_features), (C.c_void_p * n)(*[w.ctypes.data for w in ws]),
                             (C.c_void_p * n)(*[b.ctypes.data for b in bs]), vw, C.c_float(vb))
        self.__del__()              # (destroys the previous handle)
        self._h = h
        self.obs_size = int(ws[0].shape[1])
        self.obs_words = (self.obs_size + 31) // 32
        self.out_features = out_features
        self.num_actions = out_features[-1]
        self._key = (policy, weights_version(policy))

    def refresh(self, policy: torch.nn.Module, after: torch.cuda.Stream | None = None) -> bool:
        """Makes the handle hold `policy`'s current weights.  Nothing happens while it holds this very module at the same
        weights_version (a version alone cannot tell two modules apart); else the weights are loaded in place where the handle can
        (TensorCorePolicy.can_load), or the C handle is recreated with the same settings, on the current stream and after the pending work
        of stream `after` when given.  Returns True when it was recreated: CUDA graphs captured with the handle hold the old one and must be
        captured again."""
        if self._key[0] is policy and self._key[1] == weights_version(policy):
            return False
        if after is not None:
            torch.cuda.current_stream(self.device).wait_stream(after)
        if self.can_load(policy):
            self.load_weights(policy)
            return False
        self._create(policy)
        return True

    def can_load(self, policy: torch.nn.Module) -> bool:
        return False                # (FusedPolicy has no in-place load)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                getattr(lib(), self._destroy_fn)(h)
            except Exception:
                pass

    def forward_bits(self, obs_bits: torch.Tensor, probs: torch.Tensor | None = None, logits: torch.Tensor | None = None,
                     values: torch.Tensor | None = None):
        """obs_bits int32 [B, obs_words] (BatchedEnv.observe_bits / step_bits) -> softmax action weights f32 [B, A]
        (and the value head's output f32 [B] into `values` when given)."""
        assert obs_bits.is_cuda and obs_bits.element_size() == 4 and obs_bits.is_contiguous() and obs_bits.shape[-1] == self.obs_words
        B = obs_bits.numel() // self.obs_words
        if probs is None and logits is None and values is None:
            probs = torch.empty((B, self.num_actions), dtype=torch.float32, device=obs_bits.device)
        for t in (probs, logits):
            assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == B * self.num_actions)
        assert values is None or (self.has_value and values.dtype == torch.float32 and values.is_contiguous() and values.numel() == B)
        st = C.c_void_p(torch.cuda.current_stream(obs_bits.device).cuda_stream)
        check(getattr(lib(), self._forward_fn)(self._h, _dptr(obs_bits), B, _dptr(probs), _dptr(logits), _dptr(values), st))
        return probs if probs is not None else (logits if logits is not None else values)


class FusedPolicy(_PolicyHandle):
    _forward_fn, _destroy_fn = "qg_policy_forward_bits_value", "qg_policy_destroy"

    def __init__(self, policy: torch.nn.Module, device=None, with_value: bool = False):
        """with_value: also evaluate the value head (forward_bits(..., values=...)); needs the simple head layout (simple_value_head).
        refresh() recreates the handle on every weight change: it has no in-place load."""
        super().__init__(policy, device, with_value)

    def _new_handle(self, *args):
        h = C.c_void_p()
        check(lib().qg_policy_create_value(self.device_index, *args, C.byref(h)))
        return h


class TensorCorePolicy(_PolicyHandle):
    """The same network for large batches on tcgen05 tensor cores (`qg_policy_tc_*`, csrc/qg_policy_tc.cu): packed observation bits in,
    softmax action weights / logits / values out; f16 hi+lo split operands with f32 accumulation.
    Error contract (u = 2^-24, M = the forward pass on |W|, |b|, |x| without ReLU): logits and values within u (4 M + F) of a float64
    emulation of the split arithmetic, F the inputs whose lo half is an f16 subnormal (0 < h < 2^-3) forward-propagated through |W|; against
    the float64 module add the propagated split error (|v - hi - lo| <= 2^-22 |v| + 2^-25).  tests/test_policy_tc_envelope.py derives both."""

    _forward_fn, _destroy_fn = "qg_policy_tc_forward_bits", "qg_policy_tc_destroy"

    def __init__(self, policy: torch.nn.Module, max_batch: int, device=None, with_value: bool = True, training: bool = False):
        """training: also allocate the backward pass (forward_train); the handle then runs one kernel per layer."""
        if training and not with_value:
            raise NotImplementedError("TensorCorePolicy(training=True) needs the value head (with_value=True)")
        self.max_batch, self.training, self._per_layer = int(max_batch), bool(training), bool(training)
        super().__init__(policy, device, with_value)

    def _new_handle(self, *args):
        h = C.c_void_p()
        check(lib().qg_policy_tc_create(self.device_index, *args, self.max_batch, C.byref(h)))
        return h

    def _create(self, policy: torch.nn.Module):
        super()._create(policy)
        if self.training:
            check(lib().qg_policy_tc_enable_training(self._h))
        self.set_per_layer(self._per_layer)

    def _device_params(self, policy: torch.nn.Module):
        """The module's action-path weights / biases (and value head) when they can be read in place: f32, contiguous, on this device, with the
        shapes of creation; else None."""
        layers = action_layers(policy)
        if len(layers) != len(self.out_features) or int(layers[0].in_features) != self.obs_size:
            return None
        if [int(l.out_features) for l in layers] != self.out_features:
            return None
        ts = [l.weight for l in layers] + [l.bias for l in layers]
        head = simple_value_head(policy) if self.has_value else None
        if self.has_value:
            if head is None:
                return None
            ts += [head.weight, head.bias]
        if any(t is None or t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous() for t in ts):
            return None
        return layers, head

    def can_load(self, policy: torch.nn.Module) -> bool:
        """Whether load_weights(policy) applies (same shapes, parameters f32 / contiguous on this device)."""
        return self._device_params(policy) is not None

    def load_weights(self, policy: torch.nn.Module) -> None:
        """Refreshes the handle's weights in place from the module's device parameters (qg_policy_tc_load_weights_dev): stream-ordered on the
        current stream, no allocation, no host round trip; CUDA graphs captured with this handle stay valid and replay the new weights."""
        got = self._device_params(policy)
        if got is None:
            raise ValueError("load_weights needs a module with the shapes of creation whose parameters are f32, contiguous and on " + str(self.device))
        layers, head = got
        n = len(layers)
        widths = (C.c_int32 * n)(*self.out_features)
        wp = (C.c_void_p * n)(*[l.weight.data_ptr() for l in layers])
        bp = (C.c_void_p * n)(*[l.bias.data_ptr() for l in layers])
        vw = C.c_void_p(head.weight.data_ptr()) if head is not None else None
        vb = C.c_void_p(head.bias.data_ptr()) if head is not None else None
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        check(lib().qg_policy_tc_load_weights_dev(self._h, self.obs_size, n, widths, wp, bp, vw, vb, st))
        self._key = (policy, weights_version(policy))

    def set_per_layer(self, per_layer: bool) -> bool:
        """Forces the one-kernel-per-layer path (True) or lets the fused three-layer kernel run where it applies (False); returns whether
        the fused kernel will run.  A handle that refresh() recreates keeps the mode."""
        self._per_layer = bool(per_layer)
        return bool(lib().qg_policy_tc_set_mode(self._h, 1 if per_layer else 0))

    def forward_train(self, policy: torch.nn.Module, obs_bits: torch.Tensor):
        """Differentiable forward of `policy` on packed observation bits int32 [B, obs_words] -> (logits [B, A], values [B, 1]), like
        policy(dense) for a BasicPolicy.  The handle is refreshed from the module first (refresh).
        backward() writes the gradients of exactly the parameters of action_layers and simple_value_head, computed by the tcgen05 backward
        pass (qg_policy_tc_backward); autograd accumulates them into .grad.  A backward after a newer forward on this handle raises."""
        if not self.training:
            raise ValueError("forward_train needs a handle created with training=True")
        self.refresh(policy)
        layers = action_layers(policy)
        head = simple_value_head(policy)
        params = [l.weight for l in layers] + [l.bias for l in layers] + [head.weight, head.bias]
        return _TensorCoreTrain.apply(self, obs_bits, *params)


class _TensorCoreTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tcp, obs_bits, *params):
        B = obs_bits.shape[0]
        if B > tcp.max_batch:
            raise ValueError(f"forward_train: {B} rows exceed the handle's max_batch {tcp.max_batch}")
        logits = torch.empty((B, tcp.num_actions), dtype=torch.float32, device=obs_bits.device)
        values = torch.empty((B,), dtype=torch.float32, device=obs_bits.device)
        tcp.forward_bits(obs_bits, logits=logits, values=values)
        ctx.tcp, ctx.h, ctx.generation, ctx.B = tcp, tcp._h, int(lib().qg_policy_tc_generation(tcp._h)), B
        ctx.shapes = [p.shape for p in params]
        return logits, values.reshape(B, 1)

    @staticmethod
    def backward(ctx, dlogits, dvalues):
        tcp, B = ctx.tcp, ctx.B
        if tcp._h is not ctx.h:         # (a new handle counts its forwards afresh: its generation cannot tell)
            raise ValueError("backward after refresh() recreated the handle")
        dev = tcp.device
        dl = dlogits.float().contiguous() if dlogits is not None else torch.zeros((B, tcp.num_actions), dtype=torch.float32, device=dev)
        dv = dvalues.float().reshape(B).contiguous() if dvalues is not None else None
        grads = [torch.empty(s, dtype=torch.float32, device=dev) for s in ctx.shapes]
        n = len(tcp.out_features)
        gw = (C.c_void_p * n)(*[g.data_ptr() for g in grads[:n]])
        gb = (C.c_void_p * n)(*[g.data_ptr() for g in grads[n:2 * n]])
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        check(lib().qg_policy_tc_backward(tcp._h, ctx.generation, B, _dptr(dl), _dptr(dv), gw, gb, C.c_void_p(grads[2 * n].data_ptr()),
                                          C.c_void_p(grads[2 * n + 1].data_ptr()), st))
        return (None, None, *grads)


def pack_obs_bits(obs: torch.Tensor) -> torch.Tensor:
    """Dense 0/1 observation [B, ...] -> packed int32 [B, ceil(obs/32)] (host-side helper for tests and tools)."""
    flat = (obs.reshape(obs.shape[0], -1) != 0).cpu().numpy()
    B, n = flat.shape
    words = (n + 31) // 32
    pad = np.zeros((B, words * 32), dtype=bool)
    pad[:, :n] = flat
    packed = np.packbits(pad.reshape(B, words, 32), axis=2, bitorder="little").view(np.uint32).reshape(B, words)
    return torch.from_numpy(packed.view(np.int32).copy())
