"""The f32 fused policy (qg_policy_forward_bits_value: csrc/qg_policy.cu + csrc/qg_policy_kernels.cuh) over its whole shape range,
bit for bit against a CPU restatement of its arithmetic, and the one-launch search (qg_search_run) at the shapes the two-launch search
is pinned by.

Restatement (`restate`; include/qg_engine.h, qg_policy_create, states the same order)
  layer 0   q = rint(w 2^shift) (ties to even) over the transposed first layer, value column included when the network has one layer;
            shift = min(30 - e, 120) with 2^(e-1) <= max|w| < 2^e, 30 when every weight is 0.  Exact int64 sums over the set entries,
            h = fl(b + fl(fl(sum) 2^-shift)), ReLU unless it is the last layer.
  layer l   width N (value column counted), stride = N rounded up to 4, kt = max(1, 8192 // stride): the inputs k are read in tiles of kt
            rows and split by their position u = k mod kt within the tile over G chains (chain c takes u = c, c + G, ..):
              N > 256:     G = 2,  chain 0 starts from the bias;        z = c0 + c1
              65..256:     G = 4,  chain 0 starts from the bias;        z = ((c0 + c1) + c2) + c3
              N <= 64:     G = 16, every chain starts from 0;           z = ((((0 + c0) + c1) + ..) + c15) + b
            every step of a chain is one IEEE fused multiply-add (fma32), every combine one f32 add; ReLU unless it is the last layer.
  value     column A of the last layer, not part of the softmax.

fma32 emulates fmaf exactly in float64: the product of two f32 is exact; s = p + c is rounded to f32 with a correction only where s
lands exactly on an f32 midpoint and the TwoSum error of p + c says on which side the exact value lies.

Module bound (`module_bound`): the restatement (and so the kernel) against the float64 module, u = 2^-24,
  E_0 = Q + 3u (M_0 + Q) + tiny,  Q = (set entries) 2^-(shift+1)      quantisation, one rounding of the sum, the bias add
  E_l = |W_l| E_(l-1) + g_l (|b_l| + |W_l| (|h_(l-1)| + E_(l-1)))     g_l = gamma(longest chain + G): every term passes at most that many
                                                                      roundings; h = the module's activations (ReLU is 1-Lipschitz)
  plus 2^-36 of the magnitude per layer for the float64 module's own rounding and 2^-150 per rounding for subnormal results.

Softmax bound (`softmax_bound`), from the kernel's own logits: d = fl(l - max) (what the kernel computes), p* = exp(d) / sum exp(d);
  |p - p*| <= p* ((1 + 4u)(1 + u)^2 / ((1 - 4u)(1 - gamma(m))) - 1) + 2^-140,  m = ceil(A / 32) + 5 adds on any path of the lane sum and
  the butterfly, expf within 2 ulp (CUDA's documented bound: 4u relative), one IEEE division, one product; the absolute term covers
  subnormal exponentials.
"""
from __future__ import annotations

import ctypes as C
import math
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

U = 2.0 ** -24
TILE = 8192                 # kPolTileFloats
SMEM_CAP = 210 * 1024       # qg_policy_create's limit
F32, F64 = np.float32, np.float64


# ------------------------------------------------------------------------------------------------------------ exact f32 arithmetic
def fma32(a, b, c):
    """fl32(a * b + c) with a single rounding (IEEE fmaf), elementwise over broadcast f32 arrays."""
    p = np.asarray(a, F32).astype(F64) * np.asarray(b, F32).astype(F64)        # exact: 48 significant bits
    c64 = np.asarray(c, F32).astype(F64)
    s = p + c64
    bv = s - p
    e = (p - (s - bv)) + (c64 - bv)                                             # TwoSum: p + c == s + e exactly
    with np.errstate(over="ignore", invalid="ignore"):
        r = s.astype(F32)
        r64 = r.astype(F64)
        other = np.nextafter(r, np.where(s > r64, F32(np.inf), F32(-np.inf))).astype(F64)
        big = np.isinf(r64)
        mid = np.where(big, np.copysign(2.0 ** 128 - 2.0 ** 103, s), (np.where(big, 0.0, r64) + np.where(big, 0.0, other)) * 0.5)
        other = np.where(big, np.copysign(float(np.finfo(F32).max), s), other)
        fix = (s == mid) & (e != 0) & ((e > 0) == (other > np.where(big, np.copysign(np.inf, s), r64)))
    return np.where(fix, other.astype(F32), r)


def f32_of_fraction(x: Fraction) -> float:
    """x rounded to the nearest f32 (ties to even), subnormals and overflow included."""
    if x == 0:
        return 0.0
    sgn, a = (-1.0 if x < 0 else 1.0), abs(x)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    if Fraction(2) ** e > a:
        e -= 1
    q = Fraction(2) ** (max(e, -126) - 23)
    n = a / q
    m = math.floor(n)
    rem = n - m
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and m % 2 == 1):
        m += 1
    v = m * q
    if v >= Fraction(2) ** 128:
        return sgn * math.inf
    return sgn * float(v)


# ------------------------------------------------------------------------------------------------------------ networks
class Net:
    """An MLP as qg_policy_create_value takes it: W[l] f32 [out][in] (torch Linear layout), b[l], and an optional value head (vw [in of
    the last layer], vb) that the kernel evaluates as column A of the last layer."""

    def __init__(self, obs, widths, value=False, scale=1.0, mode=None, seed=0):
        rng = np.random.Generator(np.random.PCG64(seed))
        self.obs, self.A = obs, widths[-1]
        self.W, self.b = [], []
        k = obs
        for l, n in enumerate(widths):
            s = 1.0 / math.sqrt(k)
            W = rng.uniform(-s, s, (n, k))
            b = rng.uniform(-s, s, n)
            if l == 0:
                W, b = W * scale, b * scale
            self.W.append(np.ascontiguousarray(W, F32))
            self.b.append(np.ascontiguousarray(b, F32))
            k = n
        self.vw, self.vb = None, 0.0
        if value:
            k = obs if len(widths) == 1 else widths[-2]           # the value head reads the last layer's inputs
            self.vw = np.ascontiguousarray(rng.uniform(-1, 1, k) / math.sqrt(k), F32)
            self.vb = float(F32(rng.uniform(-0.1, 0.1)))
        W0 = self.W[0]
        if mode == "outlier":
            W0[0, 0] = F32(8.0 * scale)
        elif mode == "zero":
            W0[:] = 0.0
        elif mode == "tiny":                          # max |w| = 2^-101: 30 - e = 130, clamped to 120; ~9-bit q, some weights 0
            W0[:] = np.ldexp(W0 * math.sqrt(obs), -110).astype(F32)
            W0[0, 0] = F32(2.0 ** -101)
            for b in self.b:                          # biases at the same scale, so that the quantised sums reach the outputs
                b[:] = np.ldexp(b, -105).astype(F32)
            self.vb = float(np.ldexp(F32(self.vb), -105))
        elif mode == "value_outlier":                 # one layer: the value column sets the fixed-point scale
            assert len(widths) == 1 and value
            self.vw[0] = F32(16.0 * float(np.abs(W0).max()))

    def layers(self):
        """[(W f32 [N][K], b f32 [N])] as the kernel evaluates them: the value head appended to the last layer."""
        out = list(zip(self.W, self.b))
        if self.vw is not None:
            W, b = out[-1]
            out[-1] = (np.concatenate([W, self.vw[None, :]]), np.concatenate([b, np.array([self.vb], F32)]))
        return out

    def widths(self):
        return [W.shape[0] for W, _ in self.layers()]


def first_layer_shift(W0, clamp=True):
    mx = float(np.abs(W0).max())
    if mx == 0.0:
        return 30
    return min(30 - math.frexp(mx)[1], 120) if clamp else 30 - math.frexp(mx)[1]


def chain_plan(K, N, mutation=None):
    """(G, [input indices of chain c, in order]) of a dense layer with K inputs and N outputs (module docstring)."""
    stride = (N + 3) // 4 * 4
    kt = max(1, TILE // stride)
    G = 2 if N > 256 else (4 if N > 64 else 16)
    k = np.arange(K)
    if mutation == "ascending":
        return 1, [k]
    if mutation == "drop_last_row" and K % kt:
        k = k[:-1]
    grp = (k % G) if mutation == "global_group" else ((k % kt) % G)
    return G, [k[grp == c] for c in range(G)]


def dense_layer(h, W, b, relu, mutation=None):
    """One layer after the first, as the kernel computes it.  h f32 [R][K] -> f32 [R][N]."""
    R, (N, K) = h.shape[0], W.shape
    G, chains = chain_plan(K, N, mutation)
    L = max(len(c) for c in chains)
    idx = np.full((G, L), -1, np.int64)
    for c, ks in enumerate(chains):
        idx[c, :len(ks)] = ks
    acc = np.zeros((G, R, N), F32)
    if G in (1, 2, 4) or mutation == "bias_every_group":
        acc[0] = b
        if mutation == "bias_every_group":
            acc[:] = b
    for i in range(L):
        kk = idx[:, i]
        ok = kk >= 0
        ks = np.where(ok, kk, 0)
        new = fma32(W[:, ks].T[:, None, :], h[:, ks].T[:, :, None], acc)
        acc = np.where(ok[:, None, None], new, acc)
    if G == 1:
        z = acc[0]
    elif G in (2, 4):
        z = acc[0]
        for c in range(1, G):
            z = (z + acc[c]).astype(F32)
    else:
        z = np.broadcast_to(b, (R, N)).astype(F32) if mutation == "bias_first" else np.zeros((R, N), F32)
        for c in range(G):
            z = (z + acc[c]).astype(F32)
        if mutation != "bias_first":
            z = (z + b).astype(F32)
    return np.maximum(z, F32(0)) if relu else z


def restate(net: Net, x, mutation=None):
    """The kernel's logits f32 [R][A] and values f32 [R] (None without a value head) for 0/1 rows x [R][obs]."""
    layers = net.layers()
    W0, b0 = layers[0]
    shift = first_layer_shift(W0, clamp=mutation != "unclamped") - (1 if mutation == "shift" else 0)
    q = np.rint(np.ldexp(W0.astype(F64), shift)).astype(np.int64)
    acc = np.asarray(x, np.int64) @ q.T
    h = (acc.astype(F64).astype(F32) * F32(2.0 ** -shift)).astype(F32)
    h = (b0 + h).astype(F32)
    if len(layers) > 1:
        h = np.maximum(h, F32(0))
    for l, (W, b) in enumerate(layers[1:], 1):
        h = dense_layer(h, W, b, l + 1 < len(layers), mutation)
    return h[:, :net.A], (h[:, net.A] if net.vw is not None else None)


# ------------------------------------------------------------------------------------------------------------ bounds (numpy or torch)
def _t(a, dev):
    return torch.as_tensor(np.asarray(a), device=dev).double()


def module_bound(net: Net, x, dev="cpu"):
    """(z float64 [R][N_last]: the float64 module's logits and value column, E [R][N_last]: the bound of the module docstring)."""
    layers = net.layers()
    x = x if torch.is_tensor(x) else _t(x, dev)
    x = x.double()
    h, E = x, None
    shift = first_layer_shift(layers[0][0])
    for l, (W, b) in enumerate(layers):
        W64, b64 = _t(W, x.device), _t(b, x.device)
        aW = W64.abs()
        z = h @ W64.T + b64
        if l == 0:
            M = x @ aW.T + b64.abs()
            Q = x.sum(1, keepdim=True) * 2.0 ** -(shift + 1)
            E = Q + 3 * U * (M + Q) + 2.0 ** -36 * M + 2.0 ** -140
        else:
            N, K = W.shape
            G, chains = chain_plan(K, N)
            m = max(len(c) for c in chains) + G + 1
            g = m * U / (1 - m * U)
            mag = b64.abs() + (h.abs() + E) @ aW.T
            E = E @ aW.T + (g + 2.0 ** -36) * mag + m * 2.0 ** -150       # (+ the absolute error of subnormal results)
        h = torch.relu(z) if l + 1 < len(layers) else z
    return z, E


def softmax_bound(logits):
    """(p* float64, bound) for the probabilities from the kernel's logits (torch f32 [R][A])."""
    A = logits.shape[1]
    mx = logits.max(dim=1, keepdim=True).values
    d = (logits - mx).double()                      # f32 subtraction, as the kernel does it
    e = torch.exp(d)
    p = e / e.sum(dim=1, keepdim=True)
    m = -(-A // 32) + 5
    gm = m * U / (1 - m * U)
    rel = (1 + 4 * U) * (1 + U) ** 2 / ((1 - 4 * U) * (1 - gm)) - 1
    return p, p * rel + 2.0 ** -140


# ------------------------------------------------------------------------------------------------------------ observations
def make_obs(rng, B, obs, density):
    """uint8 [B][obs]: random rows at `density`, with an empty, a full and a one-hot row first."""
    x = (rng.random((B, obs)) < density).astype(np.uint8)
    if B > 0:
        x[0] = 0
    if B > 1:
        x[1] = 1
    if B > 2:
        x[2] = 0
        x[2, rng.integers(obs)] = 1
    return x


def pack(x, garbage=False):
    """uint8 [B][obs] -> uint32 [B][ceil(obs / 32)], bit i % 32 of word i // 32; garbage: the bits past obs set (the kernel masks them)."""
    B, obs = x.shape
    OW = (obs + 31) // 32
    pad = np.zeros((B, OW * 32), np.uint8)
    pad[:, :obs] = x
    if garbage:
        pad[:, obs:] = 1
    return np.ascontiguousarray(np.packbits(pad, axis=1, bitorder="little").view(np.uint32))


def emulated_rows(B, rng, most=64):
    """Row 0, the last row, the whole last CTA (8 rows) and random rows, at most `most`."""
    if B == 0:
        return np.zeros(0, np.int64)
    rows = {0, B - 1} | set(range((B - 1) // 8 * 8, B))
    free = most - len(rows)
    if free > 0 and B > len(rows):
        rows |= set(rng.choice(B, size=min(free, B), replace=False).tolist())
    return np.array(sorted(rows)[:most], np.int64)


# ------------------------------------------------------------------------------------------------------------ the envelope
# (id, obs, action-path widths (the last is A), value head, first-layer scale, first-layer mode, density, batch)
SHAPES = [
    ("w1", 81, [1, 1], False, 1.0, None, 0.3, 19),
    ("w2_value3", 81, [2, 2], True, 1.0, None, 0.3, 20),
    ("head64to65", 200, [63, 64], True, 1.0, None, 0.2, 21),              # 64 actions + value: a 65-wide head, pairs path
    ("head63to64", 200, [64, 63], True, 1.0, None, 0.2, 22),              # 63 + value: 64, narrow path
    ("pairs", 300, [65, 255, 65], False, 1.0, None, 0.2, 23),
    ("head256to257", 300, [256, 256], True, 1.0, None, 0.2, 24),          # 256 + value: consume_layer<2>
    ("head255to256", 300, [257, 255], True, 1.0, None, 0.2, 25),          # 255 + value: pairs at 256
    ("ni2", 729, [511, 512, 513, 28], False, 1.0, None, 0.04, 26),
    ("ni3_ni4", 729, [767, 768, 769, 64], True, 1.0, None, 0.04, 27),     # hidden 768: consume_layer<3>, 769: <4>; head 65: pairs
    ("ni4", 500, [1023, 1024, 100], True, 1.0, None, 0.1, 28),
    ("a1024", 64, [1024, 1023, 1024], False, 1.0, None, 0.5, 29),
    ("a1023_value", 100, [1024, 1023], True, 1.0, None, 0.5, 30),
    ("depth1", 300, [40], True, 1.0, None, 0.2, 31),
    ("depth1_w1", 300, [1], False, 1.0, None, 0.2, 32),
    ("depth1_w1024", 33, [1024], False, 1.0, None, 0.5, 33),
    ("depth1_value_scale", 300, [40], True, 1e-3, "value_outlier", 0.2, 34),
    ("depth3", 400, [300, 100, 50], True, 1.0, None, 0.1, 35),
    ("depth8", 128, [96, 80, 300, 70, 200, 64, 130, 40], True, 1.0, None, 0.3, 36),
    ("depth8_wide", 60, [1024, 1024, 769, 1024, 600, 1024, 513, 50], False, 1.0, None, 0.3, 37),
    # K at tile_rows multiples +-1 (odd kt: which chain owns an input shifts from tile to tile)
    ("kt27", 90, [55, 300, 28], False, 1.0, None, 0.3, 38),               # out 300: kt 27, K 55 = 2 kt + 1; then 300 = kt(28) + 8
    ("kt81", 90, [161, 100, 80, 100], True, 1.0, None, 0.3, 39),          # out 100: kt 81, K 161 = 2 kt - 1, later K 80 = kt - 1
    ("kt8", 90, [1024, 9, 1024, 17], False, 1.0, None, 0.3, 40),          # out 1024: kt 8, K 9 = kt + 1
    ("kt31_kt128", 90, [129, 63, 257, 16], True, 1.0, None, 0.3, 41),     # out 63: kt 128, K 129; out 257: kt 31, K 63 = 2 kt + 1
    ("kt157", 90, [315, 50, 156], True, 1.0, None, 0.3, 42),              # out 50: kt 157, K 315 = 2 kt + 1
    ("kt10", 90, [761, 768, 21], False, 1.0, None, 0.3, 43),              # out 768: kt 10, K 761 = 76 kt + 1
    # first-layer scales
    ("scale1e-3", 729, [512, 256, 28], True, 1e-3, None, 0.05, 44),
    ("scale30", 729, [512, 256, 28], True, 30.0, None, 0.05, 45),
    ("outlier", 729, [512, 256, 28], True, 0.05, "outlier", 0.05, 46),
    ("zero", 729, [512, 256, 28], True, 1.0, "zero", 0.05, 47),
    ("tiny", 500, [300, 70], True, 1.0, "tiny", 0.5, 48),
    # densities: rows whose change lists together exceed policy_ent_cap (row groups)
    ("dense1200", 1200, [600, 300, 20], True, 1.0, None, 0.5, 49),
    ("dense3000", 3000, [128, 64, 10], True, 1.0, None, 0.7, 50),
]
SHAPE_IDS = [s[0] for s in SHAPES]
MUTATIONS = ["ascending", "global_group", "bias_every_group", "bias_first", "drop_last_row", "shift", "unclamped"]


def _shape(sid):
    s = next(s for s in SHAPES if s[0] == sid)
    _, obs, widths, value, scale, mode, density, B = s
    return Net(obs, widths, value=value, scale=scale, mode=mode, seed=B), density, B


# ------------------------------------------------------------------------------------------------------------ CPU tests
def _fma_exact(a, b, c):
    return f32_of_fraction(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def test_fma_emulation_is_exact():
    """fma32 against exact rational arithmetic: random operands and the hard cases (ties, double-rounding traps, subnormal results,
    cancellation, products near the f32 range)."""
    rng = np.random.Generator(np.random.PCG64(1))
    n = 3000
    a = (rng.standard_normal(n) * np.exp2(rng.integers(-30, 30, n))).astype(F32)
    b = (rng.standard_normal(n) * np.exp2(rng.integers(-30, 30, n))).astype(F32)
    c = (rng.standard_normal(n) * np.exp2(rng.integers(-60, 60, n))).astype(F32)
    c[::3] = (-(a[::3].astype(F64) * b[::3].astype(F64))).astype(F32)            # cancellation: c ~ -a b
    cases = [
        (1.0, 2.0 ** -24, 1.0),                                                    # exact tie: to even (1)
        (1.0, 3 * 2.0 ** -24, 1.0),                                                # exact tie: to even (1 + 2^-22)
        (1 + 2.0 ** -12, 1 - 2.0 ** -12 + 2.0 ** -24, 2.0 ** 24),                  # float64 sum lands on the midpoint, exact value above
        (-(1 + 2.0 ** -12), 1 - 2.0 ** -12 + 2.0 ** -24, -(2.0 ** 24)),            # ... mirrored
        (1 + 2.0 ** -20, 1 - 2.0 ** -20, 2.0 ** 24),                               # ... below (2^24 + 1 - 2^-40)
        (1 + 2.0 ** -20, 1 - 2.0 ** -20, -(2.0 ** 24) - 2.0),                      # midpoint from the other side
        (2.0 ** -70, 1.5 * 2.0 ** -70, 2.0 ** -140),                               # subnormal results
        (2.0 ** -75, 2.0 ** -75, -(2.0 ** -149)),
        (1.25 * 2.0 ** -100, 2.0 ** -49, 2.0 ** -149),                             # a tie between subnormals
        (2.0 ** 64 * 1.5, 2.0 ** 63 * 1.25, -(2.0 ** 127)),                        # products near the top of the range
        (float(np.finfo(F32).max), 1.0, float(np.finfo(F32).max) * 2.0 ** -24),    # overflow exactly at the boundary midpoint
        (float(np.finfo(F32).max), 1.0, float(np.finfo(F32).max) * 2.0 ** -25),
        (3.0, 1.0 / 3.0, -1.0),
        (0.1, 10.0, -1.0),
    ]
    ca, cb, cc = (np.array([x[i] for x in cases], F32) for i in range(3))
    a, b, c = np.concatenate([a, ca]), np.concatenate([b, cb]), np.concatenate([c, cc])
    got = fma32(a, b, c)
    for i in range(len(a)):
        want = _fma_exact(a[i], b[i], c[i])
        assert float(got[i]) == want, (i, a[i], b[i], c[i], float(got[i]), want)
    with np.errstate(over="ignore"):
        naive = (a.astype(F64) * b.astype(F64) + c.astype(F64)).astype(F32)
    assert np.count_nonzero(naive[-len(cases):] != got[-len(cases):]) >= 3            # the traps are traps


def test_tiny_shape_engages_the_shift_clamp():
    """The "tiny" shape's first layer lies below the clamp: 30 - e exceeds 120, so the clamp sets the shift, the weights keep few bits
    and some quantise to zero (the mutation test shows that an unclamped shift changes its outputs)."""
    net, _, _ = _shape("tiny")
    W0 = net.layers()[0][0]
    assert 30 - math.frexp(float(np.abs(W0).max()))[1] > 120 and first_layer_shift(W0) == 120
    q = np.abs(np.rint(np.ldexp(W0.astype(F64), 120)))
    assert np.count_nonzero(q == 0) > 0 and np.median(q) < 2 ** 12


def test_chain_plan_partitions_every_input_once():
    for K, N in ((1, 1), (55, 300), (161, 100), (9, 1024), (1024, 17), (315, 50), (761, 768), (1024, 1024)):
        for mutation in (None, "global_group"):
            G, chains = chain_plan(K, N, mutation)
            ks = np.sort(np.concatenate(chains))
            assert np.array_equal(ks, np.arange(K)) and all(np.all(np.diff(c) > 0) for c in chains)


@pytest.mark.parametrize("sid", SHAPE_IDS)
def test_restatement_within_bound_of_float64_module(sid):
    """The restatement means the module: within the derived bound of the float64 forward pass of the same weights."""
    net, density, _ = _shape(sid)
    rng = np.random.Generator(np.random.PCG64(3))
    x = make_obs(rng, 10, net.obs, density)
    lg, val = restate(net, x)
    z, E = module_bound(net, x)
    got = np.concatenate([lg, val[:, None]], 1) if val is not None else lg
    err = np.abs(got.astype(F64) - z.numpy())
    assert np.all(err <= E.numpy()), (sid, float((err / E.numpy()).max()))


def test_restatement_matches_basic_policy_module():
    """Net and the float64 bound mean what FusedPolicy hands the kernel: the same weights taken from a BasicPolicy give the module's
    float64 output."""
    from qiskit_gym_b200.policy import action_layers, simple_value_head
    from qiskit_gym_b200.search import BasicPolicy
    torch.manual_seed(4)
    pol = BasicPolicy([9, 9], 12, embedding_size=96, common_layers=(70,)).eval()
    net = Net(81, [96, 70, 12], value=True)
    for i, l in enumerate(action_layers(pol)):
        net.W[i] = np.ascontiguousarray(l.weight.detach().numpy(), F32)
        net.b[i] = np.ascontiguousarray(l.bias.detach().numpy(), F32)
    v = simple_value_head(pol)
    net.vw, net.vb = np.ascontiguousarray(v.weight.detach().numpy().reshape(-1), F32), float(v.bias.detach()[0])
    x = make_obs(np.random.Generator(np.random.PCG64(2)), 12, 81, 0.3)
    with torch.no_grad():
        lg, val = pol.double()(torch.from_numpy(x).double())
    z, E = module_bound(net, x)
    assert torch.allclose(z[:, :12], lg, rtol=0, atol=1e-13) and torch.allclose(z[:, 12], val[:, 0], rtol=0, atol=1e-13)   # (BLAS order)
    rl, rv = restate(net, x)
    assert np.all(np.abs(rl - lg.numpy()) <= E[:, :12].numpy()) and np.all(np.abs(rv - val[:, 0].numpy()) <= E[:, 12].numpy())


@pytest.mark.parametrize("mutation", MUTATIONS)
def test_mutations_change_a_logit_bit(mutation):
    """Each plausible kernel bug, applied to the restatement, changes at least one logit or value bit at a shape the GPU test runs, so
    the bit-exact comparison would catch it."""
    rng = np.random.Generator(np.random.PCG64(6))
    hits = []
    for sid in SHAPE_IDS:
        net, density, _ = _shape(sid)
        x = make_obs(rng, 12, net.obs, density)
        a, av = restate(net, x)
        b, bv = restate(net, x, mutation=mutation)
        if np.any(a.view(np.uint32) != b.view(np.uint32)) or (av is not None and np.any(av.view(np.uint32) != bv.view(np.uint32))):
            hits.append(sid)
            if len(hits) >= 2:
                break
    assert hits, mutation


def test_value_column_in_softmax_breaks_the_probability_bound():
    """Counting the value column in the softmax moves probabilities outside the softmax bound the GPU test applies."""
    net, density, _ = _shape("head256to257")
    x = make_obs(np.random.Generator(np.random.PCG64(8)), 12, net.obs, density)
    lg, val = restate(net, x)
    p, bound = softmax_bound(torch.from_numpy(lg))
    wrong = torch.softmax(torch.from_numpy(np.concatenate([lg, val[:, None]], 1)).double(), dim=1)[:, :net.A]
    assert torch.any((wrong - p).abs() > bound)


# ------------------------------------------------------------------------------------------------------------ GPU: the kernel
def _lib():
    from qiskit_gym_b200._lib import lib
    return lib()


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class Handle:
    """A raw qg_policy (any depth 1..8, with or without a value head) created from a Net through the C ABI."""

    def __init__(self, net: Net, device=0, layers=None):
        L = _lib()
        ws = [net.W[i] for i in range(len(net.W))] if layers is None else [w for w, _ in layers]
        bs = list(net.b) if layers is None else [b for _, b in layers]
        n = len(ws)
        self._keep = (ws, bs, net.vw)
        h = C.c_void_p()
        self.rc = L.qg_policy_create_value(device, net.obs, n, (C.c_int32 * n)(*[w.shape[0] for w in ws]),
                                           (C.c_void_p * n)(*[w.ctypes.data for w in ws]), (C.c_void_p * n)(*[b.ctypes.data for b in bs]),
                                           None if net.vw is None else net.vw.ctypes.data_as(C.c_void_p), C.c_float(net.vb), C.byref(h))
        self.h = h if self.rc == 0 else None
        self.net = net

    def forward(self, bits, B, probs=None, logits=None, values=None):
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc = _lib().qg_policy_forward_bits_value(self.h, _ptr(bits), B, _ptr(probs), _ptr(logits), _ptr(values), st)
        torch.cuda.synchronize()
        return rc

    def __del__(self):
        if getattr(self, "h", None):
            _lib().qg_policy_destroy(self.h)
            self.h = None


def _run(net, x, garbage=False, dev=torch.device("cuda", 0)):
    """(probs, logits, values or None) of the kernel for rows x."""
    h = Handle(net)
    assert h.rc == 0, _lib().qg_last_error().decode()
    B = x.shape[0]
    bits = torch.from_numpy(pack(x, garbage).view(np.int32)).to(dev)
    probs = torch.empty((B, net.A), dtype=torch.float32, device=dev)
    logits = torch.empty_like(probs)
    values = torch.empty(B, dtype=torch.float32, device=dev) if net.vw is not None else None
    assert h.forward(bits, B, probs, logits, values) == 0, _lib().qg_last_error().decode()
    return probs, logits, values


def _check(net, x, rng, probs, logits, values, most=64):
    """Emulated rows bit for bit; every row within the module bound (logits, value) and the softmax bound (probs)."""
    B = x.shape[0]
    dev = logits.device
    rows = emulated_rows(B, rng, most)
    rl, rv = restate(net, x[rows])
    kl = logits[torch.from_numpy(rows).to(dev)].cpu().numpy()
    bad = np.argwhere(kl != rl)
    assert bad.size == 0, ("logit bits", bad[:5], kl[tuple(bad[0])], rl[tuple(bad[0])])
    if values is not None:
        kv = values[torch.from_numpy(rows).to(dev)].cpu().numpy()
        assert np.array_equal(kv == rv, np.ones_like(kv, bool)), ("value bits", np.argwhere(kv != rv)[:5])
    for s in range(0, B, 16384):                       # every row against the float64 module
        xs = torch.from_numpy(x[s:s + 16384]).to(dev)
        z, E = module_bound(net, xs, dev)
        got = logits[s:s + 16384].double()
        if values is not None:
            got = torch.cat([got, values[s:s + 16384].double()[:, None]], 1)
        assert torch.all((got - z).abs() <= E), ("module bound", float(((got - z).abs() / E).max()))
        p, pb = softmax_bound(logits[s:s + 16384])
        assert torch.all((probs[s:s + 16384].double() - p).abs() <= pb), ("softmax bound", float(((probs[s:s + 16384].double() - p).abs() / pb).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("sid", SHAPE_IDS)
def test_kernel_equals_restatement(sid):
    net, density, B = _shape(sid)
    rng = np.random.Generator(np.random.PCG64(B))
    x = make_obs(rng, B * 3, net.obs, density)
    probs, logits, values = _run(net, x)
    _check(net, x, rng, probs, logits, values)


def _max_obs(widths):
    """The largest obs_size qg_policy_create accepts for these widths (bisection on the C ABI)."""
    lo, hi = 1, 65535
    while lo < hi:
        mid = (lo + hi + 1) // 2
        h = Handle(Net(mid, widths, value=True, seed=1))
        if h.rc == 0:
            lo = mid
        else:
            assert h.rc == -3, h.rc                                   # QG_ERR_UNSUPPORTED: shared memory
            hi = mid - 1
    return lo


@pytest.mark.gpu
def test_observation_sizes_to_the_shared_memory_limit():
    widths = [64, 10]
    top = _max_obs(widths)
    # the plan of policy_smem_bytes (qg_policy_kernels.cuh) at 2..4 weight stages: obs_size is capped by it, well below 65535
    def plan(obs, stages):
        ow, cap = (obs + 31) // 32, (obs if obs > 2048 else min(8 * obs, 2048))
        b = (stages * TILE + 2 * 64 * 8 + 1024 * 8) * 4 + (2 * stages + 2) * 8 + 2 * 8 * ow * 4 + 128 + cap * 4
        return (b + 127) // 128 * 128
    assert any(plan(top, s) <= SMEM_CAP < plan(top + 1, s) for s in (2, 3, 4)), top
    assert top < 65535
    assert Handle(Net(top + 1, widths, value=True, seed=1)).rc == -3
    for obs in (1, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049, top):
        net = Net(obs, widths, value=True, seed=obs)
        rng = np.random.Generator(np.random.PCG64(obs))
        x = make_obs(rng, 43, obs, 0.5)
        x[3:6] = 1                                      # full rows: every row's list fills the entry capacity alone
        probs, logits, values = _run(net, x, garbage=True)
        _check(net, x, rng, probs, logits, values, most=24)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 61, 62, 63, 64, 65, 66, 67, 68, 200, 65536 + 77])
def test_batch_sizes(B):
    """Every tail size of the last CTA, an MCTS-sized batch and a collector batch: a row's outputs do not depend on B."""
    net = Net(729, [512, 256, 28], value=True, seed=5)
    rng = np.random.Generator(np.random.PCG64(B))
    x = make_obs(rng, B, 729, 0.04)
    if B == 0:
        h = Handle(net)
        bits = torch.zeros((1, 23), dtype=torch.int32, device="cuda")
        probs = torch.full((1, 28), 7.0, device="cuda")
        assert h.forward(bits, 0, probs, None, None) == 0 and torch.all(probs == 7.0)
        return
    probs, logits, values = _run(net, x)
    _check(net, x, rng, probs, logits, values)


@pytest.mark.gpu
def test_output_subsets_and_sentinels():
    """probs only, logits only, values only: the same bits as all three together, and nothing written past row B."""
    net = Net(300, [256, 64], value=True, seed=9)
    rng = np.random.Generator(np.random.PCG64(9))
    B, pad = 37, 11
    x = make_obs(rng, B, 300, 0.2)
    dev = torch.device("cuda", 0)
    bits = torch.from_numpy(pack(x).view(np.int32)).to(dev)
    h = Handle(net)
    sentinel = float.fromhex("0x1.5555p-3")
    outs = {k: torch.full((B + pad,) + ((net.A,) if k != "values" else ()), sentinel, device=dev) for k in ("probs", "logits", "values")}
    assert h.forward(bits, B, outs["probs"], outs["logits"], outs["values"]) == 0
    for k in outs:
        one = torch.full_like(outs[k], sentinel)
        assert h.forward(bits, B, *[one if j == k else None for j in ("probs", "logits", "values")]) == 0
        assert torch.equal(one[:B].view(torch.int32), outs[k][:B].view(torch.int32)), k
        assert torch.all(one[B:] == sentinel) and torch.all(outs[k][B:] == sentinel), k
    _check(net, x, rng, outs["probs"][:B], outs["logits"][:B], outs["values"][:B])


@pytest.mark.gpu
def test_refusals():
    dev = torch.device("cuda", 0)
    deep = Net(50, [16] * 9, seed=2)
    assert Handle(deep).rc == -1                                        # 9 layers: QG_ERR_INVALID
    assert Handle(Net(50, [16, 1025], seed=2)).rc == -3                 # width 1025: QG_ERR_UNSUPPORTED
    assert Handle(Net(50, [16, 1024], value=True, seed=2)).rc == -3     # 1024 + the value column
    assert Handle(Net(50, [1025], seed=2)).rc == -3
    for bad in (np.nan, np.inf, -np.inf):
        net = Net(50, [16, 4], seed=2)
        net.W[0][3, 7] = bad
        assert Handle(net).rc == -1                                     # non-finite first-layer weights: QG_ERR_INVALID
    plain = Handle(Net(50, [16, 4], seed=2))
    bits = torch.zeros((8, 2), dtype=torch.int32, device=dev)
    values = torch.zeros(8, device=dev)
    assert plain.forward(bits, 8, None, None, values) == -1             # values without a value head
    assert plain.forward(bits, 8, None, None, None) == -1               # no output at all
    assert plain.forward(bits, -1, torch.zeros((8, 4), device=dev), None, None) == -1


# ------------------------------------------------------------------------------------------------------------ GPU: one-launch search
def _search_pair(name, emb, common, R, max_depth, deterministic, scramble, seed=2):
    """(fused, persistent) results of the same search: key, solution, returns (f32 bits), final states, per-env remaining depths and
    steps played, per-CTA decision counts (fused: derived from the steps played, persistent: the kernel's own)."""
    from oracle import oracle as orc
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch
    from tests import helpers as H
    kind, n, gs, kw = H.config_table()[name]
    kw = dict(kw)
    if kind != H.PAULI:
        kw["add_inverts"] = False
    torch.manual_seed(seed)
    probe = orc.OracleEnv(kind, n, gs, add_perms=False, **kw)
    pol = BasicPolicy(probe.obs_shape(), len(gs), embedding_size=emb, common_layers=common)
    t = H.random_targets(kind, n, gs, 1, seed, scramble=scramble, **({"num_rotations": 2} if kind == H.PAULI else {}))
    state = t[0, : H.payload_lengths(kind, n, t)[0]].tolist()
    out = {}
    for backend in ("fused", "persistent"):
        rs = RolloutSearch(kind, n, gs, pol, R, max_depth=max_depth, policy_backend=backend, use_cuda_graph=False, **kw)
        if backend == "persistent":
            rs.check_supported()
        res = rs.solve(state, deterministic=deterministic, seed=5, first_rollout_id=1000)
        depth = rs.env.status()[3].cpu().numpy().copy()
        played = np.zeros((R + 7) // 8 * 8, np.int64)          # steps each rollout took: the length of its action log
        played[:R] = [len(a) for a in rs.env.solutions()]
        if backend == "persistent":
            dec = rs._decisions.cpu().numpy()[: (R + 7) // 8].copy()
        else:                                                   # a CTA decides until its 8 rollouts are final or the budget is spent
            dec = np.maximum(1, np.minimum(played.reshape(-1, 8).max(1), max_depth)).astype(np.int32)
        out[backend] = (res.key, res.actions, rs.env.returns().cpu().numpy().view(np.uint32).copy(),
                        [rs.env.get_state(b) for b in sorted({0, 7, 8, R // 2, R - 1})], np.concatenate([depth, played]), dec)
        del rs
    return out["fused"], out["persistent"]


def _assert_same_search(a, b):
    assert a[0] == b[0] and a[1] == b[1]
    assert np.array_equal(a[2], b[2])
    assert all(np.array_equal(x, y) for x, y in zip(a[3], b[3]))
    assert np.array_equal(a[4], b[4])
    assert np.array_equal(a[5], b[5])


@pytest.mark.gpu
@pytest.mark.parametrize("name,emb,common,R,max_depth,deterministic,scramble", [
    ("C1_perm_grid3", 1024, (32,), 200, 10, False, 4),                              # first layer 1024 wide, B mod 8 = 0
    ("lf5_line_swap", 600, (32,), 201, 10, True, 6),                                # 513..1024, tail 1
    ("clifford3_allgates", 64, (1024, 600, 300, 100, 64, 70), 202, 8, False, 6),    # 8 layers, hidden wider than 512, tail 2
    ("lf40_line", 513, (64,), 203, 5, False, 400),                                  # dense 1600-entry rows: the fresh pass groups rows
    ("clifford16_allgates", 256, (128,), 204, 4, True, 400),
    ("clifford20_line", 128, (700,), 205, 4, False, 400),
    ("pauli6_line", 777, (200, 65), 206, 10, False, 6),
    ("C1_perm_grid3", 64, (32,), 207, 2, True, 8),                                   # budget exit: max_depth below the rollouts' length
    ("lf5_line_swap", 1000, (1000,), 15, 3, False, 12),
])
def test_persistent_search_equals_two_kernel_search_envelope(name, emb, common, R, max_depth, deterministic, scramble):
    a, b = _search_pair(name, emb, common, R, max_depth, deterministic, scramble)
    _assert_same_search(a, b)


# ------------------------------------------------------------------------------------------------------------ shared-memory limit of qg_search_run
def _perm_search(edges, R=16, backend="persistent", max_depth=4):
    """A Permutation search with a SWAP per edge and a BasicPolicy(64, (32,)); None where the policy itself does not fit
    (qg_policy_create refuses it)."""
    from qiskit_gym_b200.search import BasicPolicy, RolloutSearch
    from tests import helpers as H
    n, gs = H.gateset_from_coupling_map(edges, ("SWAP",))
    torch.manual_seed(1)
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(32,))
    try:
        return RolloutSearch(H.PERM, n, gs, pol, R, max_depth=max_depth, policy_backend=backend, use_cuda_graph=False, add_inverts=False)
    except NotImplementedError:
        return None


def _refusal(rs):
    """None when the zero-decision probe accepts, else (bytes needed, dynamic, static, bytes allowed) from its QG_ERR_UNSUPPORTED message."""
    try:
        rs.check_supported()
        return None
    except NotImplementedError as e:
        m = re.search(r"need (\d+) bytes of shared memory \((\d+) dynamic \+ (\d+) static\), one block may have (\d+)", str(e))
        assert m, str(e)
        return tuple(int(v) for v in m.groups())


def _pairs(n, count=None):
    p = [(i, j) for i in range(n) for j in range(i + 1, n)]
    return p if count is None else p[:count]


@pytest.mark.gpu
def test_search_shared_memory_check_counts_the_action_weights():
    """A Permutation with hundreds of SWAPs: the policy and the step region fit the old check (policy + step <= 220 KB), but the CTA's
    action weights (8 x A floats) take the launch past one block's limit.  The probe refuses it, RLSynthesis falls back to the PyTorch
    policy and solves; the pair with the most actions the probe accepts runs and equals the two-launch search; one action more is
    refused.  (45 qubits with all 990 SWAPs is such a pair at 3 weight stages; 64 qubits with 1000 SWAPs at 2, where the policy plan is
    32 KB smaller.)"""
    window = None
    for n, edges in ((45, _pairs(45)), (64, _pairs(64, 1000))):
        rs = _perm_search(edges)
        if rs is None:
            continue
        r = _refusal(rs)
        A = len(edges)
        del rs
        if r is not None and r[1] - 8 * A * 4 <= 220 * 1024:          # dynamic - action weights = policy + step: what the old check saw
            window = (n, edges, r)
            break
    assert window is not None, "no pair between the old and the corrected limit: the probe accepts a search that cannot launch"
    n, edges, (need, dyn, stat, limit) = window
    assert need == dyn + stat and need > limit and limit >= 227 * 1024 and stat >= 9 * 4          # s_active + s_ret[8]

    # RLSynthesis picks the PyTorch policy for it, and that search solves a target one SWAP from the identity
    from oracle import oracle as orc
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    spec = SynthSpec.from_coupling_map("PermutationEnv", edges, basis_gates=("SWAP",), max_depth=8)
    rls = RLSynthesis(spec, {}, {"embedding_size": 64, "common_layers": [32]})
    state = list(range(n))
    a, b = edges[len(edges) // 2]
    state[a], state[b] = state[b], state[a]
    got = rls.solve(state, num_searches=16384, seed=1)
    assert rls._searches[16384].backend == "torch"
    assert got is not None and len(got) >= 1
    kind, _, gs, kw = rls._env_args(add_perms=False)
    chk = orc.OracleEnv(kind, n, gs, add_inverts=False, add_perms=False)
    chk.set_state(state)
    for act in got:
        chk.step(act)
    assert chk.success()
    del rls

    # the most actions the probe accepts on these qubits: that pair runs and equals "fused"; one action more is refused
    lo, hi = n, len(edges) - 1
    rs = _perm_search(edges[:lo])
    assert _refusal(rs) is None
    del rs
    while lo < hi:
        mid = (lo + hi + 1) // 2
        rs = _perm_search(edges[:mid])
        if _refusal(rs) is None:
            lo = mid
        else:
            hi = mid - 1
        del rs
    rs = _perm_search(edges[:lo + 1])
    r = _refusal(rs)
    assert r is not None and 0 < r[0] - r[3] <= 8 * 4 + 2 * 8 * 4 + 128      # one action: its weights, two activation rows, the plan's rounding
    del rs
    state = list(range(n))
    for a, b in (edges[1], edges[lo // 2]):
        state[a], state[b] = state[b], state[a]
    out = []
    for backend in ("fused", "persistent"):
        rs = _perm_search(edges[:lo], R=21, backend=backend)
        res = rs.solve(state, deterministic=False, seed=3)
        out.append((res.key, res.actions, rs.env.returns().cpu().numpy().view(np.uint32).copy(), rs.env.status()[3].cpu().numpy().copy(),
                    [len(x) for x in rs.env.solutions()]))
        del rs
    assert out[0][0] == out[1][0] and out[0][1] == out[1][1]
    assert np.array_equal(out[0][2], out[1][2]) and np.array_equal(out[0][3], out[1][3]) and out[0][4] == out[1][4]
