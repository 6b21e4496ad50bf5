"""The tensor-core policy (TensorCorePolicy, csrc/qg_policy_tc.cu) over its whole shape envelope and at collector batch sizes, against two
float64 references with error bounds derived from its arithmetic.

References
  module     pol.double()(dense.double()): what the f32 module means, evaluated in float64.
  emulation  what the kernel says it computes (qg_policy_tc.cu, header): a weight or hidden activation v is carried as hi = half(v),
             lo = half(v - hi) (torch .half() rounds to nearest-even, like __float2half_rn); a product is a_hi*w_hi + a_hi*w_lo + a_lo*w_hi
             (layer 1: a is 0 / 1, exact, so x*w_hi + x*w_lo), summed in float64, rounded to f32, + f32 bias, ReLU on hidden layers.

Magnitude  M = the forward pass on |W|, |b| and |x| without ReLU (float64).  Every |partial sum| of every layer is <= M of that layer.
u = 2^-24 (f32 unit roundoff).

Bound against the emulation: |kernel - emulation| <= u (C_EMUL M + F), C_EMUL = 4,
  F_1 = 0,  F_l = |W_l| F_(l-1) + |W_l| s_(l-1),  s = [0 < h < 2^-3] of the emulation's hidden activation h.
  The two do the same split and the same products; they differ only in how the sum is accumulated: float64 in the emulation, the
  f32 accumulator in tensor memory in the kernel, and in the split the next layer makes of the slightly different activation.
  C_EMUL M: a worst-case bound is 2u per rounding times the partial sum; summed over the n K = 16 MMA issues of a layer (up to 96) that
  is ~200 u M or more, looser than the error of the precision bugs this file has to catch (dropping a_hi*w_lo for one K block moves a
  logit by ~2^-12 of one K block's partial sum, tens of u M).  The bound instead uses that the partial sums of these networks are sums
  of terms of both signs: for K terms they are ~sqrt(K) smaller than M at every layer (K >= 64 after padding), and n rounding errors
  of varying sign add like sqrt(n), so sqrt(n) * e * M / sqrt(K) <= e M for n <= 3 K / 16, with e the error of one issue relative to
  its partial sum.  e = 4u: the adder aligns the 16 products and the accumulator to the largest exponent and normalises the sum, each
  step truncating (at most 2u).  (One round-to-nearest per issue, e = 2u, is what the CPU restatement below models; the B200 measures
  up to 2.2 u M against the emulation — on the two-layer network with a 512-wide head and on the value column at weight scale 30 — so
  its accumulator is not that: the constant counts both truncations.)
  F: an activation that differs by a few ulp can round to a lo one step away: 2^-22 |h| (counted in C_EMUL) or, once lo is an f16
  subnormal (|h| < 2^-3), 2^-24 absolute — u per such input, times |w| — which dominates for small weights (scale 1e-2: activations
  ~1e-4).  (An activation the emulation has at 0 that the kernel computes as a tiny positive value is that value — at most the
  propagated error — exactly split to 2^-25: it is covered by the propagation, not by s.)
  test_simulated_accumulator_within_emulation_bound restates the accumulator (f32 rounding after every K = 16 issue, to nearest and
  toward zero) on the CPU and checks it against this bound at several shapes and scales.

Bound against the module: |kernel - module| <= u (C_EMUL M + F) + R, R = the representation error forward-propagated:
  R_1 = 4u |W_1| |x| + 2^-25 (1 . |x|) + 2u M_1
  R_l = |W_l| R_(l-1) + 12u |W_l| M_(l-1) + 2^-25 (1 . M_(l-1)) + 2^-25 |W_l| 1 + 2u M_l
  from  v = hi + lo + r,  |r| <= 2^-22 |v| + 2^-25  (2^-25: half the spacing of f16 subnormals, where lo lands for |v| < 2^-3 — the
  default init's weights already), so that a*w - (a_hi w_hi + a_hi w_lo + a_lo w_hi) = a_hi r_w + r_a w + a_lo w_lo + a_lo r_w
  <= 3 * 2^-22 |a||w| + 2^-25 (|a| + |w|) (to first order; layer 1: a exact, 2^-22 |w| + 2^-25 per active entry), plus the f32 rounding
  of the sum and of the bias add (u each).  The absolute 2^-25 term is what makes weights of ~1e-3 carry ~2e-5 M of error: it is
  derived, not a fudge, and it is what the module comparison at scale 1e-2 exercises.

Softmax: with the logits of a row within e of the reference, |p - p_ref| <= min(1, p_ref ((exp(2e) - 1) + (A + 8) 2u) + 2^-120)
  (shift invariance; expf 2 ulp, A-term f32 sum, one division, one product; the absolute term covers f32 underflow).
"""
import numpy as np
import pytest
import torch

U = 2.0 ** -24
SUB = 2.0 ** -25          # f16 subnormal half-spacing: the absolute part of the split's representation error
C_EMUL = 4.0
KB = 64                   # the kernels' K block


# ----------------------------------------------------------------------------------------------- reference machinery (CPU and GPU)
def net_params(pol, with_value=True):
    """[(W f32 [N, K], b f32 [N])] of the action path; with_value appends the value head as one more row of the last layer (as the
    kernels do: column A of the head)."""
    from qiskit_gym_b200.policy import action_layers, simple_value_head
    ps = [(l.weight.detach().float().clone(), l.bias.detach().float().clone()) for l in action_layers(pol)]
    if with_value:
        v = simple_value_head(pol)
        W, b = ps[-1]
        ps[-1] = (torch.cat([W, v.weight.detach().float().reshape(1, -1)]), torch.cat([b, v.bias.detach().float().reshape(1)]))
    return ps


def split(t):
    """f32 tensor -> (hi, lo) as float64: hi = half(v), lo = half(v - hi) (the difference is exact in f32)."""
    hi = t.half()
    lo = (t - hi.float()).half()
    return hi.double(), lo.double()


def emulate(params, x, drop_hilo=None, act_hi_only=False, shift=None, hidden=None):
    """The kernel's arithmetic in float64 (module docstring).  x: 0/1 float64 [B, obs].  Returns f32 [B, N_last] (pre-softmax).
    Mutations (CPU tests only): drop_hilo=(layer, kb) drops a_hi*w_lo of K block kb of that layer; act_hi_only drops every a_lo;
    shift=(layer, k) makes input column k of that layer read the weights of column k + 1 (a one-position image column shift).
    hidden: a list that receives every hidden layer's f32 activations."""
    h = x
    L = len(params)
    for l, (W, b) in enumerate(params):
        W = W.to(x.device)
        if shift is not None and shift[0] == l:
            W = W.clone()
            W[:, shift[1]] = W[:, shift[1] + 1]
        whi, wlo = split(W)
        if drop_hilo is not None and drop_hilo[0] == l:
            wlo = wlo.clone()
            wlo[:, drop_hilo[1] * KB:(drop_hilo[1] + 1) * KB] = 0.0
        if l == 0:
            acc = h @ whi.T + h @ wlo.T
        else:
            ahi, alo = split(h)
            if act_hi_only:
                alo = torch.zeros_like(alo)
            acc = ahi @ whi.T + ahi @ wlo.T + alo @ whi.T
        z = acc.float() + b.to(x.device)
        h = torch.relu(z) if l + 1 < L else z
        if hidden is not None and l + 1 < L:
            hidden.append(h)
    return h


def magnitudes(params, x):
    """[M_1, ..., M_L]: the forward pass on |W|, |b|, |x| without ReLU (float64)."""
    out, h = [], x.abs()
    for W, b in params:
        h = h @ W.to(x.device).double().abs().T + b.to(x.device).double().abs()
        out.append(h)
    return out


def flip_bound(params, hidden):
    """F of the module docstring (unscaled: the bound is u F), from the emulation's hidden activations."""
    F = torch.zeros_like(hidden[0], dtype=torch.float64)
    for l, (W, b) in enumerate(params[1:], 1):
        aW = W.to(F.device).double().abs()
        h = hidden[l - 1].double().abs()
        F = F @ aW.T + ((h > 0) & (h < 0.125)).double() @ aW.T
    return F


def representation_bound(params, x, Ms):
    """R of the module docstring: the emulation's distance from the float64 module, forward-propagated."""
    R = None
    for l, (W, b) in enumerate(params):
        aW = W.to(x.device).double().abs()
        if l == 0:
            R = 4 * U * (x.abs() @ aW.T) + SUB * x.abs().sum(1, keepdim=True) + 2 * U * Ms[0]
        else:
            Mp = Ms[l - 1]
            R = R @ aW.T + 12 * U * (Mp @ aW.T) + SUB * Mp.sum(1, keepdim=True) + SUB * aW.sum(1)[None, :] + 2 * U * Ms[l]
    return R


def module_ref(pol, dense):
    """float64 module on the policy's device: (logits [B, A], value [B])."""
    with torch.no_grad():
        p64 = _double_copy(pol)
        lg, v = p64(dense.to(next(p64.parameters()).device).double())
    return lg, v.reshape(-1)


def _double_copy(pol):
    import copy
    return copy.deepcopy(pol).double()


def softmax_bound(p_ref, logit_err):
    """|p - p_ref| bound from a per-entry logit error bound (module docstring)."""
    A = p_ref.shape[1]
    e = logit_err.max(dim=1, keepdim=True).values
    b = p_ref * torch.expm1(2 * e).clamp(max=1.0) + p_ref * (A + 8) * 2 * U + 2.0 ** -120
    return b.clamp(max=1.0)                 # (a probability error is at most 1: where the logit bound exceeds 1/2 the check is vacuous)


class Refs:
    """Both references and both bounds for one network on one set of dense observations."""

    def __init__(self, pol, dense, with_value=True, params=None):
        dev = dense.device
        self.A = action_layers_out(pol)
        self.params = params if params is not None else net_params(pol, with_value)
        x = dense.reshape(dense.shape[0], -1).double()
        hid = []
        self.emul = emulate(self.params, x, hidden=hid).double()
        Ms = magnitudes(self.params, x)
        self.M = Ms[-1]
        self.b_emul = U * (C_EMUL * self.M + flip_bound(self.params, hid))
        self.b_mod = self.b_emul + representation_bound(self.params, x, Ms)
        lg, v = module_ref(pol, dense)
        self.mod = torch.cat([lg, v[:, None]], 1) if with_value else lg
        self.mod = self.mod.to(dev)
        A = self.A
        self.p_emul = torch.softmax(self.emul[:, :A], 1)
        self.p_mod = torch.softmax(self.mod[:, :A], 1)
        self.bp_emul = softmax_bound(self.p_emul, self.b_emul[:, :A])
        self.bp_mod = softmax_bound(self.p_mod, self.b_mod[:, :A])

    def check(self, B, logits=None, probs=None, values=None, tag=""):
        """Every row < B of the given outputs within both bounds of both references."""
        A = self.A
        for name, got, col in (("logits", logits, slice(0, A)), ("values", values, A)):
            if got is None:
                continue
            g = got.double().reshape(B, -1) if name == "logits" else got.double().reshape(B)
            for ref, bnd, which in ((self.emul, self.b_emul, "emulation"), (self.mod, self.b_mod, "module")):
                r, bb = ref[:B, col], bnd[:B, col]
                err = (g - r).abs()
                assert torch.isfinite(g).all(), (tag, name)
                ratio = float((err / bb).max())
                assert ratio <= 1.0, (tag, name, which, ratio, float(err.max()))
        if probs is not None:
            g = probs.double().reshape(B, A)
            for ref, bnd, which in ((self.p_emul, self.bp_emul, "emulation"), (self.p_mod, self.bp_mod, "module")):
                ratio = float(((g - ref[:B]).abs() / bnd[:B]).max())
                assert ratio <= 1.0, (tag, "probs", which, ratio)


def action_layers_out(pol):
    from qiskit_gym_b200.policy import action_layers
    return int(action_layers(pol)[-1].out_features)


def scale_policy(pol, s):
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(s)
    return pol


def make_policy(obs, A, emb, common, seed, scale=1.0, policy_layers=(), value_layers=()):
    from qiskit_gym_b200.search import BasicPolicy
    torch.manual_seed(seed)
    return scale_policy(BasicPolicy([obs], A, embedding_size=emb, common_layers=common, policy_layers=policy_layers,
                                    value_layers=value_layers).eval(), scale)


def random_dense(rng, B, obs, density):
    d = (rng.random((B, obs)) < density).astype(np.float32)
    if B > 2:
        d[0] = 0.0                      # an empty observation and a full one
        d[1] = 1.0
    return torch.from_numpy(d)


# ----------------------------------------------------------------------------------------------- CPU: the reference machinery itself
def test_split_representation_error():
    """hi + lo carries v to 2^-22 |v| + 2^-25 (the bound the module comparison is derived from), across normal and subnormal lo."""
    g = torch.Generator().manual_seed(0)
    for s in (30.0, 1.0, 0.05, 1e-3, 1e-5):
        v = (torch.rand(100000, generator=g) * 2 - 1) * s
        hi, lo = split(v)
        r = (v.double() - hi - lo).abs()
        assert bool((r <= 2.0 ** -22 * v.double().abs() + SUB).all()), s
        assert float(lo.abs().max()) <= 2.0 ** -11 * float(v.abs().max()) * 1.001 + SUB
    assert split(torch.tensor([1.0]))[1].item() == 0.0


def _simulated_kernel(params, x, rz):
    """The kernel's accumulator restated: products of the split halves, f32 accumulation rounded after every K = 16 issue, in the
    kernels' issue order (K block, k slice, hi*hi, hi*lo, lo*hi).  rz: round toward zero instead of to nearest."""
    def rnd(v):
        f = v.float()
        if rz:
            over = f.double().abs() > v.abs()
            f = torch.where(over, torch.nextafter(f, torch.zeros_like(f)), f)
        return f.double()
    h = x
    L = len(params)
    for l, (W, b) in enumerate(params):
        whi, wlo = split(W)
        K = W.shape[1]
        Kp = (K + KB - 1) // KB * KB
        pad = lambda t: torch.nn.functional.pad(t, (0, Kp - t.shape[1]))
        whi, wlo = pad(whi), pad(wlo)
        if l == 0:
            terms = [(pad(h), whi), (pad(h), wlo)]
        else:
            ahi, alo = split(h)
            terms = [(pad(ahi), whi), (pad(ahi), wlo), (pad(alo), whi)]
        acc = torch.zeros(x.shape[0], W.shape[0], dtype=torch.float64)
        for k0 in range(0, Kp, 16):
            for a, w in terms:
                acc = rnd(acc + a[:, k0:k0 + 16] @ w[:, k0:k0 + 16].T)
        z = acc.float() + b
        h = torch.relu(z) if l + 1 < L else z
    return h


CPU_SHAPES = [  # obs, A, emb, common, scale, density
    (64, 8, 128, (64,), 1.0, 0.5),
    (25, 8, 512, (256,), 1.0, 0.3),
    (81, 14, 256, (128,), 1e-2, 0.2),
    (36, 27, 200, (100,), 30.0, 0.5),
    (9, 1, 128, (64,), 1.0, 0.5),
]


@pytest.mark.parametrize("rz", [False, True])
def test_simulated_accumulator_within_emulation_bound(rz):
    """The f32 accumulator of the kernels, restated (round to nearest and toward zero), stays within C_EMUL u M of the emulation, and the
    emulation within R of the float64 module — the two derivations of the module docstring, checked where no GPU is needed."""
    rng = np.random.Generator(np.random.PCG64(11))
    for i, (obs, A, emb, common, scale, dens) in enumerate(CPU_SHAPES):
        pol = make_policy(obs, A, emb, common, seed=i, scale=scale)
        x = random_dense(rng, 300, obs, dens).double()
        ps = net_params(pol)
        hid = []
        e = emulate(ps, x, hidden=hid).double()
        Ms = magnitudes(ps, x)
        sim = _simulated_kernel(ps, x, rz).double()
        r = float(((sim - e).abs() / (U * (C_EMUL * Ms[-1] + flip_bound(ps, hid)))).max())
        assert r <= 0.5, (i, r)                     # with margin: the hardware's accumulator may differ from this restatement
        lg, v = module_ref(pol, x.float())
        mod = torch.cat([lg, v[:, None]], 1)
        rm = float(((e - mod).abs() / representation_bound(ps, x, Ms)).max())
        assert rm <= 1.0, (i, rm)


def _mutation_setup():
    # obs 64 -> 128 -> 128 -> 8 + value: one K block of the head is half of its K
    pol = make_policy(64, 8, 128, (128,), seed=5)
    x = random_dense(np.random.Generator(np.random.PCG64(12)), 1000, 64, 0.5).double()
    ps = net_params(pol)
    hid = []
    e = emulate(ps, x, hidden=hid).double()
    bound = U * (C_EMUL * magnitudes(ps, x)[-1] + flip_bound(ps, hid))
    return pol, ps, x, e, bound


@pytest.mark.parametrize("mutation", ["hilo_one_kblock", "act_hi_only", "column_shift", "padding_bias"])
def test_emulation_bound_rejects_mutations(mutation):
    """Each mutated copy of the emulation models a subtle kernel bug; the emulation bound u (C_EMUL M + F) must reject it (on some entry)."""
    pol, ps, x, e, bound = _mutation_setup()
    A = 8
    if mutation == "hilo_one_kblock":
        m = emulate(ps, x, drop_hilo=(2, 1)).double()            # the head's K block 1 of 2
    elif mutation == "act_hi_only":
        m = emulate(ps, x, act_hi_only=True).double()
    elif mutation == "column_shift":
        m = emulate(ps, x, shift=(1, 77)).double()               # one column of layer 2's image
    else:
        # the head's first padding column (A + 1: after the value column) with a non-zero bias, read as an action by the soft-max
        W, b = ps[-1]
        bad = list(ps[:-1]) + [(torch.cat([W, torch.zeros(1, W.shape[1])]), torch.cat([b, torch.tensor([0.25])]))]
        lg = emulate(bad, x).double()
        p_bad = torch.softmax(torch.cat([lg[:, :A], lg[:, A + 1:]], 1), 1)[:, :A]
        p_ok = torch.softmax(e[:, :A], 1)
        assert float(((p_bad - p_ok).abs() / softmax_bound(p_ok, bound[:, :A])).max()) > 1.0
        return
    assert float(((m - e).abs() / bound).max()) > 1.0


# ----------------------------------------------------------------------------------------------- GPU: shape envelope, small batches
SMALL_B = (1, 127, 128, 129, 1000)
SENTINEL = -7.25

# fused shapes, pairwise over E x C (every pair once), A and obs spread over them, value head on / off:
#   (obs, A, E, C, value).  E 200 pads to 256, C 100 to 128; NC = E_pad / 128 in {1, 2, 3, 4}, H = round_up(A + value, 16) in 16..128
FUSED = [
    (9, 1, 128, 64, True), (25, 3, 128, 100, False), (36, 8, 128, 192, True), (64, 14, 128, 256, False),
    (81, 15, 200, 64, False), (256, 27, 200, 100, True), (729, 28, 200, 192, False), (9, 49, 200, 256, True),
    (25, 63, 384, 64, True), (36, 64, 384, 100, False), (64, 72, 384, 192, True), (81, 104, 384, 256, False),
    (256, 124, 512, 64, False), (729, 126, 512, 100, True), (9, 127, 512, 192, False), (36, 127, 512, 256, True),
]
# per-layer-only shapes: (obs, A, E, common, policy_layers, value)
PER_LAYER = [
    (81, 12, 300, (256,), (), True),              # E = 300: 64-wide column tiles (NT = 64)
    (64, 14, 1260, (128,), (), True),             # E = 1260: n_tiles = 10 of 128
    (25, 8, 4096, (64,), (), False),              # a 4096-wide layer
    (36, 27, 512, (), (), True),                  # 2 layers
    (64, 40, 256, (192, 128), (), True),          # 4 layers
    (81, 20, 256, (128,), (64,), False),          # policy_layers, no value head
]


def _dev():
    return torch.device("cuda", 0)


def _sentinel_outputs(B, A, has_value, pad=64):
    """Views [:B] of buffers max_batch + pad long, filled with a sentinel."""
    dev = _dev()
    lb = torch.full(((B + pad) * A,), SENTINEL, device=dev)
    pb = torch.full(((B + pad) * A,), SENTINEL, device=dev)
    vb = torch.full((B + pad,), SENTINEL, device=dev) if has_value else None
    return lb, pb, vb


def _run(tcp, bits, B, A, has_value, outs=("logits", "probs", "values")):
    """forward_bits into sentinel-filled views; asserts nothing past row B changed; returns the outputs (or None)."""
    lb, pb, vb = _sentinel_outputs(B, A, has_value)
    kw = {}
    if "logits" in outs:
        kw["logits"] = lb[:B * A].view(B, A)
    if "probs" in outs:
        kw["probs"] = pb[:B * A].view(B, A)
    if "values" in outs and has_value:
        kw["values"] = vb[:B]
    tcp.forward_bits(bits[:B].contiguous(), **kw)
    torch.cuda.synchronize()
    for buf, n in ((lb, B * A), (pb, B * A), (vb, B)):
        if buf is not None:
            assert bool((buf[n:] == SENTINEL).all()), "wrote past the batch"
    return (kw.get("logits"), kw.get("probs"), kw.get("values"))


def _bits(dense):
    from qiskit_gym_b200.policy import pack_obs_bits
    return pack_obs_bits(dense).to(_dev())


def _i32(ts):
    return [None if t is None else t.view(torch.int32).clone() for t in ts]


def _check_network(pol0, pol1, has_value, obs, expect_fused, Bs, density, rng, max_batch=None, rolls=()):
    """Both modes, every batch in Bs: both references and bounds, writes past the batch, output combinations (largest B), two calls
    bit-identical, row independence under the given rolls, and load_weights (P0 -> P1 -> P0) against fresh handles."""
    from qiskit_gym_b200.policy import TensorCorePolicy
    dev = _dev()
    Bmax = max(Bs)
    A = action_layers_out(pol0)
    pol0, pol1 = pol0.to(dev), pol1.to(dev)
    dense = random_dense(rng, Bmax, obs, density).to(dev)
    bits = _bits(dense)
    refs0, refs1 = Refs(pol0, dense, has_value), Refs(pol1, dense, has_value)
    tcp = TensorCorePolicy(pol0, max_batch=max_batch or Bmax, device=dev, with_value=has_value)
    assert tcp.set_per_layer(False) == expect_fused
    modes = [False, True] if expect_fused else [True]
    first = {}
    for per_layer in modes:
        tcp.set_per_layer(per_layer)
        for B in Bs:
            out = _run(tcp, bits, B, A, has_value)
            refs0.check(B, *out, tag=(per_layer, B))
            if B == Bmax:
                first[per_layer] = _i32(out)
                again = _i32(_run(tcp, bits, B, A, has_value))
                assert all(a is None or torch.equal(a, b) for a, b in zip(first[per_layer], again)), "two calls differ"
                for one in (("logits",), ("probs",), ("values",)) if has_value else (("logits",), ("probs",)):
                    alone = _i32(_run(tcp, bits, B, A, has_value, outs=one))
                    for a, b in zip(first[per_layer], alone):
                        if b is not None:
                            assert torch.equal(a, b), (per_layer, one)
                for r in rolls:
                    rolled = _i32(_run(tcp, torch.roll(bits[:B], r, 0).contiguous(), B, A, has_value))
                    for a, b in zip(first[per_layer], rolled):
                        if a is not None:
                            assert torch.equal(torch.roll(a, r, 0), b), ("row independence", per_layer, r)
    # load_weights: P0 -> P1 equals a fresh handle of P1; P1 -> P0 equals the original outputs (padding untouched)
    tcp.load_weights(pol1)
    fresh = TensorCorePolicy(pol1, max_batch=max_batch or Bmax, device=dev, with_value=has_value)
    for per_layer in modes:
        tcp.set_per_layer(per_layer)
        fresh.set_per_layer(per_layer)
        got, want = _run(tcp, bits, Bmax, A, has_value), _run(fresh, bits, Bmax, A, has_value)
        for a, b in zip(_i32(got), _i32(want)):
            if a is not None:
                assert torch.equal(a, b), ("load_weights != fresh", per_layer)
        refs1.check(Bmax, *got, tag=("P1", per_layer))
    tcp.load_weights(pol0)
    for per_layer in modes:
        tcp.set_per_layer(per_layer)
        back = _i32(_run(tcp, bits, Bmax, A, has_value))
        for a, b in zip(first[per_layer], back):
            if a is not None:
                assert torch.equal(a, b), ("P0 reloaded", per_layer)


@pytest.mark.gpu
@pytest.mark.parametrize("obs,A,E,C,value", FUSED)
def test_fused_shape_envelope(obs, A, E, C, value):
    rng = np.random.Generator(np.random.PCG64(obs * 1000 + A))
    p0 = make_policy(obs, A, E, (C,), seed=A)
    p1 = make_policy(obs, A, E, (C,), seed=A + 1000, scale=0.3)
    _check_network(p0, p1, value, obs, True, SMALL_B, 0.3 if obs > 64 else 0.5, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("obs,A,E,common,pl,value", PER_LAYER)
def test_per_layer_shape_envelope(obs, A, E, common, pl, value):
    rng = np.random.Generator(np.random.PCG64(E + A))
    p0 = make_policy(obs, A, E, common, seed=A, policy_layers=pl)
    p1 = make_policy(obs, A, E, common, seed=A + 1000, scale=3.0, policy_layers=pl)
    _check_network(p0, p1, value, obs, False, SMALL_B, 0.4, rng)


CHECKPOINTS = [("clifford_3q_custom", 36, 8), ("lf_5_line", 25, 8), ("perm_square_3x3", 81, 12)]


def _checkpoint(name, obs, A):
    import os
    from qiskit_gym_b200.search import BasicPolicy
    pol = BasicPolicy([obs], A)
    sd = torch.load(os.path.join(os.path.dirname(__file__), "golden", "models", name + ".pt"), map_location="cpu", weights_only=True)
    pol.load_state_dict(sd)
    return pol.eval()


@pytest.mark.gpu
@pytest.mark.parametrize("name,obs,A", CHECKPOINTS)
@pytest.mark.parametrize("scale", [1.0, 1e-2, 30.0])
def test_trained_checkpoints_and_scales(name, obs, A, scale):
    """The repository's trained checkpoints (obs < 64: a partly filled first K block), plain and scaled, through the tensor-core policy in
    both modes and through FusedPolicy (f32 FFMA) against the float64 module.  Scale 30 saturates the soft-max."""
    from qiskit_gym_b200.policy import FusedPolicy
    rng = np.random.Generator(np.random.PCG64(obs))
    p0 = scale_policy(_checkpoint(name, obs, A), scale)
    p1 = make_policy(obs, A, 512, (256,), seed=obs, scale=scale)          # default init at the same scale, for load_weights
    _check_network(p0, p1, True, obs, True, SMALL_B, 0.3, rng)
    # FusedPolicy: f32 FFMA sums of K terms (fixed-point first layer): recursive-summation bound 2 K u per layer on M, plus R
    dev = _dev()
    dense = random_dense(rng, 1000, obs, 0.3).to(dev)
    fp = FusedPolicy(p0.to(dev), device=dev, with_value=True)
    lg, pr, v = torch.empty(1000, A, device=dev), torch.empty(1000, A, device=dev), torch.empty(1000, device=dev)
    fp.forward_bits(_bits(dense), probs=pr, logits=lg, values=v)
    x = dense.double()
    ps = net_params(p0)
    Ms = magnitudes(ps, x)
    bound = 2 * U * sum(W.shape[1] for W, _ in ps) * Ms[-1]
    lm, vm = module_ref(p0, dense)
    got = torch.cat([lg.double(), v.double()[:, None]], 1)
    ref = torch.cat([lm, vm[:, None]], 1)
    assert float(((got - ref).abs() / bound).max()) <= 1.0
    assert float(((pr.double() - torch.softmax(lm, 1)).abs() / softmax_bound(torch.softmax(lm, 1), bound[:, :A])).max()) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("obs,A,E,common,value", [
    (64, 128, 512, (256,), True),          # 129 head columns
    (64, 8, 4097, (256,), True),           # a width of 4097
    (64, 8, 512, (4097,), False),
])
def test_refusals(obs, A, E, common, value):
    from qiskit_gym_b200.policy import TensorCorePolicy
    pol = make_policy(obs, A, E, common, seed=0).to(_dev())
    with pytest.raises(NotImplementedError):
        TensorCorePolicy(pol, max_batch=16, device=_dev(), with_value=value)


@pytest.mark.gpu
def test_max_batch_exceeded_and_a128_without_value():
    """A = 128 without the value head is the widest head (H = 128, fused and per-layer); a batch over max_batch is refused."""
    rng = np.random.Generator(np.random.PCG64(128))
    p0 = make_policy(64, 128, 256, (128,), seed=1)
    p1 = make_policy(64, 128, 256, (128,), seed=2, scale=0.5)
    _check_network(p0, p1, False, 64, True, (1, 129, 1000), 0.5, rng)
    from qiskit_gym_b200.policy import TensorCorePolicy
    tcp = TensorCorePolicy(p0.to(_dev()), max_batch=100, device=_dev(), with_value=False)
    bits = _bits(random_dense(rng, 101, 64, 0.5))
    with pytest.raises(ValueError):
        tcp.forward_bits(bits)


# ----------------------------------------------------------------------------------------------- GPU: collector batch sizes
COLLECTOR_SHAPES = {   # name: (obs, A, E, common, fused)
    "C3": (256, 72, 512, (256,), True),
    "C2_lf8_line": (64, 14, 512, (256,), True),      # the default config, A = 14: the staged (A % 4 != 0) head
    "NC3_C192": (49, 27, 384, (192,), True),
    "per_layer": (81, 12, 300, (256,), False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(COLLECTOR_SHAPES))
def test_collector_batch_sizes(name):
    """Multi-tile CTAs (persistent grids of min(tiles, SMs) CTAs): every row at B around and past one wave, against both references;
    two calls identical; rows rolled by 1 and 129 give the same per-row bits; load_weights at this batch."""
    obs, A, E, common, fused = COLLECTOR_SHAPES[name]
    S = torch.cuda.get_device_properties(0).multi_processor_count
    Bs = (S * 128 - 1, S * 128, S * 128 + 1, 3 * S * 128 + 77, 65536)
    rng = np.random.Generator(np.random.PCG64(len(name)))
    p0 = make_policy(obs, A, E, common, seed=7)
    p1 = make_policy(obs, A, E, common, seed=8, scale=2.0)
    _check_network(p0, p1, True, obs, fused, Bs, 0.3, rng, max_batch=65537, rolls=(1, 129))


# ----------------------------------------------------------------------------------------------- GPU: the collector end to end at scale
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2_lf8_line", "C3_clifford8_full"])
def test_collect_packed_at_scale(name):
    """collect_packed with the default policy shape (512 -> [256]) at B = 2 S 128 + 77 (3 waves of row tiles, a partial last tile), T = 3:
    ~200 envs re-enacted with the oracle (first, last, the envs on either side of CTA-wave and tile boundaries, random ones), the
    probabilities the collector sampled from within the module bound of the float64 module, and graph replay equal to eager."""
    from qiskit_gym_b200 import BatchedEnv
    from qiskit_gym_b200.collector import RolloutCollector
    from qiskit_gym_b200.search import BasicPolicy
    from tests import helpers as H
    from tests.test_collector_packed import reenact, rollout_fields
    S = torch.cuda.get_device_properties(0).multi_processor_count
    B, T, seed, first, gamma, lam = 2 * S * 128 + 77, 3, 31, 3, 0.99, 0.9
    kind, n, gs, kw = H.config_table()[name]
    ekw = dict(kw, add_inverts=False, add_perms=False, difficulty=2, max_depth=5, depth_slope=2)
    envs = [BatchedEnv(kind, n, gs, B, **ekw) for _ in range(2)]
    torch.manual_seed(0)
    pol = BasicPolicy(envs[0].obs_shape(), len(gs))
    cols = [RolloutCollector(e, pol, gamma=gamma, lam=lam, use_twists=False, seed=seed, first_env_id=first) for e in envs]
    ro = cols[0].collect_packed(T, use_cuda_graph=False)
    rng = np.random.Generator(np.random.PCG64(2))
    rows = {0, B - 1, 127, 128, 129}
    for w in (1, 2):
        rows |= {w * S * 128 - 1, w * S * 128}
    rows |= set(int(k) * 128 + d for k in rng.integers(1, B // 128, size=40) for d in (-1, 0))
    rows |= set(int(r) for r in rng.integers(0, B, size=200 - len(rows)))
    rows = sorted(rows)
    probs = cols[0]._packed[(T, False)]["probs"]
    obs = ro.unpack_obs()
    for t in range(T):
        Refs(pol, obs[t, rows].float()).check(len(rows), probs=probs[t, rows].contiguous(), tag=t)
    reenact(ro, (kind, n, gs, ekw), cols[0]._tcp, None, None, seed, first, T, B, gamma, lam, rows=rows)
    # graph: the second rollout of a graph collector (captured, replayed) equals the second eager rollout
    eager = rollout_fields(cols[0].collect_packed(T, use_cuda_graph=False))
    cols[1].collect_packed(T, use_cuda_graph=True)
    graph = rollout_fields(cols[1].collect_packed(T, use_cuda_graph=True))
    assert cols[1]._packed[(T, False)]["graph"] is not None
    for a, b in zip(eager, graph):
        assert torch.equal(a, b)
