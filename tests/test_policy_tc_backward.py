"""The tensor-core backward pass (TensorCorePolicy.forward_train, qg_policy_tc_backward in csrc/qg_policy_tc.cu) against two float64
references, with error bounds derived from its arithmetic in the style of test_policy_tc_envelope.py (whose split, net_params, magnitudes,
flip_bound and representation_bound are reused here).

Arithmetic (what the kernels say they compute).  Layers l = 0 .. L-1 (0-based), H_l = the input of layer l (H_0 = the 0/1 observation,
H_l = relu(z_(l-1))), dZ_l = the gradient at layer l's pre-activation; the head's dZ is [dlogits, dvalues] (column A = the value head).
  scales   s_(L-1) = 15 - e with amax(dZ_head) < 2^e; going down, b_(l-1) = b_l colsum_l (colsum_l = max_k sum_n |W_l[n][k]|, inflated by
           2^-9) and s_(l-1) from b_(l-1) the same way: every scaled |dZ| stays below 2^15 (no f16 overflow), and its halves are normal f16
           wherever |dZ| is within ~2^14 of the bound.  dZ_l is carried as the split of the f32 value dZ_l 2^s_l.
  dgrad    dZ_(l-1) 2^s_(l-1) = mask_l * f32(zhi whi + zhi wlo + zlo whi) 2^(s_(l-1) - s_l), mask_l = (hi | lo of H_l) != 0
  wgrad    dW_l = 2^-s_l f32-sum over 1024-row chunks, in chunk order, of (zhi^T hhi + zhi^T hlo + zlo^T hhi)   (layer 0: zhi^T x + zlo^T x)
  db       db_l = 2^-s_l sum over chunks of the chunk's sum of (zhi + zlo)
The emulation below evaluates exactly these in float64 (sums unrounded, one f32 rounding where the kernel leaves f32).

Magnitude  G: the backward pass on |dZ_head|, |W| and |H| without masks: GZ_(L-1) = |dZ_head|, GZ_(l-1) = GZ_l |W_l|, G_dW_l = GZ_l^T |H_l|,
G_db_l = sum_rows GZ_l.  Every |partial sum| of the kernels (unscaled) is at most G of its output.  u = 2^-24.

Bound against the emulation (E_l: the bound on |dZ_l kernel - dZ_l emulation|, E_(L-1) = 0):
  dgrad accumulator   C_EMUL u G_dH (G_dH = GZ_l |W_l|), with the forward's argument and constant: the products dZ w have both signs like
                      the forward's a w, and K (= the layer's width) is the forward's range; + u G_dH for the f32 result.
  wgrad accumulator   K is the chunk's rows (1024, far longer than a forward K), and the products dZ h do not have to change sign (H >= 0,
                      and a value loss can push every row the same way), so no cancellation is assumed: n issues of e = 4u each (align +
                      normalise, truncating) against partial sums <= G give 4 u n G, n = terms * rows / 16 (terms = 3, layer 0: 2; rows =
                      min(batch, 1024) rounded up to 16: the zero rows past the batch add exact zeros).
  fixed-order sum     the f32 sum of the chunks, in order: u (chunks - 1) G; the db partials (8 rows sequential, a 7-level tree): 15 u G
                      <= 4 u n G;  the final 2^-s product is exact.  Together  u (4 n + chunks + 1) G.
  split of dZ         once the kernel's dZ_l differs from the emulation's (E_l > 0), its halves may round differently: 2^-22 |dZ| per half
                      pair (2^-21 G), or 2^-25 absolute in scaled units (lo an f16 subnormal) -> 2^(-24 - s_l) in gradient units (2x: the
                      scale the kernel derives from its f32 column sums may be one below the float64 one).
  inputs H            the kernel's H_l is within dH_l = u (C_EMUL M + F) of the emulation's (test_policy_tc_envelope.py), and its split
                      may flip like dZ's: dH_l + 2^-21 |H_l| + 2^-24 where dH_l > 0.
  ReLU masks          where |z_(l-1)| <= dz_(l-1) (the forward bound) the two masks may disagree: the whole G_dH there.
  so   E_(l-1) = (E_l + Phi_l) |W_l| + (C_EMUL + 1) u G_dH + G_dH [|z_(l-1)| <= dz_(l-1)]
       |dW_l - emul| <= u (4 n + chunks + 1) G_dW_l + (E_l + Phi_l)^T |H_l| + GZ_l^T (dH_l + Psi_l)
       |db_l - emul| <= u (4 n + chunks + 1) G_db_l + sum_rows (E_l + Phi_l)
  with Phi_l = [E_l > 0] (2^-21 GZ_l + 2^(-24 - s_l)), Psi_l = [dH_l > 0] (2^-21 |H_l| + 2^-24).
Bound against float64 autograd of the module: the same propagation with the forward bound widened by the envelope's representation bound R
(the emulated forward against the module), plus the split's representation error of every product, v = hi + lo + r, |r| <= 2^-22 |v| +
2^-25 (scaled units for dZ):  a w - (ahi whi + ahi wlo + alo whi) <= 3 2^-22 |a||w| + 2^-25 (|a| + |w|) to first order, i.e.
  dgrad  12 u G_dH + 2^(-25 - s_l) (1 |W_l|) + 2^-25 GZ_l 1         wgrad  12 u G_dW + 2^(-25 - s_l) 1^T |H_l| + 2^-25 GZ_l^T 1 (layer 0:
  H exact: 4 u G_dW + 2^(-25 - s_l) 1^T |H_0|)                        db  4 u G_db + rows 2^(-25 - s_l)
and the ReLU masks of the module compared where |z| is within the kernel's forward bound against the module.
"""
import math

import numpy as np
import pytest
import torch

from tests.test_policy_tc_envelope import (C_EMUL, KB, SUB, U, flip_bound, magnitudes, make_policy, net_params, random_dense,
                                           representation_bound, split)

CHUNK = 1024                 # rows per wgrad chunk (kChunkTiles x 128)


# ----------------------------------------------------------------------------------------------- reference machinery (CPU and GPU)
def forward_emul(params, x):
    """The split forward of the envelope test's emulation, keeping every layer's input H_l (x, then f32 relu(z)) and pre-activation z_l."""
    Hs, zs, h = [x], [], x
    for l, (W, b) in enumerate(params):
        whi, wlo = split(W.to(x.device))
        if l == 0:
            acc = h @ whi.T + h @ wlo.T
        else:
            ahi, alo = split(h)
            acc = ahi @ whi.T + ahi @ wlo.T + alo @ whi.T
        z = acc.float() + b.to(x.device)
        zs.append(z)
        if l + 1 < len(params):
            h = torch.relu(z)
            Hs.append(h)
    return Hs, zs


def scale_exp(b):
    if not (b > 0.0) or not math.isfinite(b):
        return 0
    return max(-100, min(100, 15 - math.frexp(b)[1]))


def scales(params, dz_head):
    """s_l of the module docstring (float64 column sums: the kernel's f32 ones may give one less, which the bound allows)."""
    b, s = float(dz_head.abs().max()), [0] * len(params)
    for l in reversed(range(len(params))):
        s[l] = scale_exp(b)
        hi, lo = split(params[l][0])
        b = float(np.float32(b) * np.float32(float((hi + lo).abs().sum(0).max()) * (1 + 2.0 ** -9)))
    return s


def backward_emul(params, Hs, dz_head, s=None, drop_hilo=None, no_scale=False, skip_bias_chunk=None, wrong_mask=False):
    """The kernels' backward in float64 (module docstring).  dz_head f32 [B, N_last].  Returns ({l: (dW f64, db f64)}, scales).
    Mutations (CPU tests only): drop_hilo=(l, kb) drops zhi*wlo of K block kb of layer l's dgrad; no_scale uses s = 0; skip_bias_chunk=c
    leaves row chunk c out of every bias gradient; wrong_mask takes the head's dgrad ReLU mask from the input of the layer below it."""
    L = len(params)
    if s is None:
        s = [0] * L if no_scale else scales(params, dz_head)
    zsc = dz_head.float() * 2.0 ** s[L - 1]
    out = {}
    for l in reversed(range(L)):
        zhi, zlo = split(zsc)
        H = Hs[l]
        if l == 0:
            hhi, hlo = H.double(), None
        else:
            hhi, hlo = split(H)
        wg = zhi.T @ hhi + zlo.T @ hhi + (zhi.T @ hlo if hlo is not None else 0.0)
        rows = zhi + zlo
        if skip_bias_chunk is not None:
            rows = rows.clone()
            rows[skip_bias_chunk * CHUNK:(skip_bias_chunk + 1) * CHUNK] = 0.0
        out[l] = (wg * 2.0 ** -s[l], rows.sum(0) * 2.0 ** -s[l])
        if l == 0:
            break
        whi, wlo = split(params[l][0].to(zsc.device))
        if drop_hilo is not None and drop_hilo[0] == l:
            wlo = wlo.clone()
            wlo[drop_hilo[1] * KB:(drop_hilo[1] + 1) * KB] = 0.0
        acc = zhi @ whi + zhi @ wlo + zlo @ whi
        mh, ml = split(Hs[l - 1 if wrong_mask and l == L - 1 else l])
        mask = (mh != 0) | (ml != 0)
        zsc = torch.where(mask, acc.float() * 2.0 ** (s[l - 1] - s[l]), torch.zeros((), device=acc.device))
    return out, s


def forward_bounds(params, x, Hs):
    """Per layer l >= 1: (kernel - emulation bound, emulation - module bound) of z_(l-1) (ReLU is 1-Lipschitz: also of H_l)."""
    Ms = magnitudes(params, x)
    emul, rep = [None], [None]
    for l in range(1, len(params)):
        F = flip_bound(params[:l], Hs[1:l]) if l > 1 else torch.zeros_like(Ms[0])
        emul.append(U * (C_EMUL * Ms[l - 1] + F))
        rep.append(representation_bound(params[:l], x, Ms[:l]))
    return emul, rep


def backward_bounds(params, x, Hs, zs, dz_head, s, module=False, kernel=True):
    """{l: (bound dW, bound db)}: against the emulation, or (module=True) against float64 autograd (module docstring).  kernel=False with
    module=True: the emulation against autograd, the representation part alone (no accumulator terms, no kernel forward error)."""
    L, B = len(params), x.shape[0]
    femul, frep = forward_bounds(params, x, Hs)
    m_tiles = -(-B // 128)
    chunks = -(-m_tiles // 8)
    rows_in_chunk = -(-min(B, CHUNK) // 16) * 16        # (the zero rows past the batch add exact zeros: no rounding)
    GZ = dz_head.double().abs()
    E = torch.zeros_like(GZ)
    out = {}
    for l in reversed(range(L)):
        H = Hs[l].double()
        aH = H.abs()
        terms = 2 if l == 0 else 3
        n = terms * rows_in_chunk // 16
        acc_c = U * (4 * n + chunks + 1) if kernel else 0.0
        Phi = torch.where(E > 0, 2.0 ** -21 * GZ + 2.0 ** (-24 - s[l]), torch.zeros((), dtype=torch.float64, device=GZ.device))
        if l > 0:
            dH = (femul[l] if kernel else 0.0) + (frep[l] if module else 0.0)
            Psi = torch.where(dH > 0, 2.0 ** -21 * aH + 2.0 ** -24, torch.zeros((), dtype=torch.float64, device=GZ.device))
            in_term = GZ.T @ (dH + Psi)
        else:
            in_term = 0.0
        bW = acc_c * (GZ.T @ aH) + (E + Phi).T @ aH + in_term
        bb = acc_c * GZ.sum(0) + (E + Phi).sum(0)
        if module:
            sub = 2.0 ** (-25 - s[l])
            if l == 0:
                bW = bW + 4 * U * (GZ.T @ aH) + sub * aH.sum(0)[None, :]
            else:
                bW = bW + 12 * U * (GZ.T @ aH) + sub * aH.sum(0)[None, :] + SUB * GZ.sum(0)[:, None]
            bb = bb + 4 * U * GZ.sum(0) + B * sub
        out[l] = (bW, bb)
        if l == 0:
            break
        aW = params[l][0].to(GZ.device).double().abs()
        GdH = GZ @ aW
        dz = (femul[l] if kernel else 0.0) + (frep[l] if module else 0.0)
        flips = (zs[l - 1].double().abs() <= dz).double()
        En = (E + Phi) @ aW + ((C_EMUL + 1) * U * GdH if kernel else 0.0) + GdH * flips
        if module:
            En = En + 12 * U * GdH + 2.0 ** (-25 - s[l]) * aW.sum(0)[None, :] + SUB * GZ.sum(1, keepdim=True)
        E, GZ = En, GdH
    return out


def module_grads(pol, dense, dlogits, dvalues):
    """float64 autograd of the module with the given upstream gradients: {l: (dW, db)} of the action path, the value head in the head row."""
    import copy
    from qiskit_gym_b200.policy import action_layers, simple_value_head
    p64 = copy.deepcopy(pol).double()
    lg, v = p64(dense.double())
    torch.autograd.backward([lg, v.reshape(-1)], [dlogits.double(), dvalues.double()])
    out = {}
    layers = action_layers(p64)
    for l, lin in enumerate(layers):
        gW, gb = lin.weight.grad, lin.bias.grad
        if l == len(layers) - 1:
            head = simple_value_head(p64)
            gW = torch.cat([gW, head.weight.grad.reshape(1, -1)])
            gb = torch.cat([gb, head.bias.grad.reshape(1)])
        out[l] = (gW, gb)
    return out


def check_grads(got, ref, bnd, tag=""):
    for l in ref:
        for name, g, r, b in (("W", got[l][0], ref[l][0], bnd[l][0]), ("b", got[l][1], ref[l][1], bnd[l][1])):
            g = g.double().to(r.device)
            assert torch.isfinite(g).all(), (tag, l, name)
            err = (g - r).abs()
            ratio = float(torch.where(err == 0, torch.zeros_like(err), err / b).max())      # (0 / 0 where G = 0: exact zeros)
            assert ratio <= 1.0, (tag, l, name, ratio)


# ----------------------------------------------------------------------------------------------- CPU: the reference machinery itself
CPU_SHAPES = [  # obs, A, emb, common, scale, density, B
    (64, 8, 128, (64,), 1.0, 0.5, 300),
    (25, 8, 256, (128,), 1.0, 0.3, 2100),
    (81, 14, 128, (64,), 1e-2, 0.2, 500),
    (36, 27, 128, (64,), 30.0, 0.5, 400),
    (9, 1, 64, (), 1.0, 0.5, 200),
]


def _case(i, shape, mean_loss=True):
    obs, A, emb, common, scale, dens, B = shape
    pol = make_policy(obs, A, emb, common, seed=i, scale=scale)
    x = random_dense(np.random.Generator(np.random.PCG64(20 + i)), B, obs, dens).double()
    g = torch.Generator().manual_seed(30 + i)
    up = torch.randn(B, A + 1, generator=g) / (B if mean_loss else 1.0)
    return pol, x, up


def test_emulation_within_representation_bound_of_autograd():
    """The emulated backward against float64 autograd of the module: within the module bound minus the kernel's accumulation part (the
    representation part alone, with the forward's representation error)."""
    for i, shape in enumerate(CPU_SHAPES):
        pol, x, up = _case(i, shape)
        ps = net_params(pol)
        Hs, zs = forward_emul(ps, x)
        em, s = backward_emul(ps, Hs, up)
        ref = module_grads(pol, x, up[:, :-1], up[:, -1])
        check_grads(em, ref, backward_bounds(ps, x, Hs, zs, up, s, module=True, kernel=False), tag=str(i))


def _simulated_backward(params, Hs, dz_head, s, rz):
    """The kernels' f32 accumulators restated: dgrad rounded after every K = 16 issue (K block, slice, hi*hi, hi*lo, lo*hi), wgrad rounded
    after every 16-row issue within 1024-row chunks, chunks summed in f32 in order.  rz: round toward zero."""
    def rnd(v):
        f = v.float()
        if rz:
            over = f.double().abs() > v.abs()
            f = torch.where(over, torch.nextafter(f, torch.zeros_like(f)), f)
        return f.double()
    L = len(params)
    zsc = dz_head.float() * 2.0 ** s[L - 1]
    out = {}
    for l in reversed(range(L)):
        zhi, zlo = split(zsc)
        H = Hs[l]
        hhi, hlo = (H.double(), None) if l == 0 else split(H)
        terms = [(zhi, hhi), (zhi, hlo), (zlo, hhi)] if hlo is not None else [(zhi, hhi), (zlo, hhi)]
        B = zhi.shape[0]
        tot_w, tot_b = None, None
        for c0 in range(0, B, CHUNK):
            accw = torch.zeros(zhi.shape[1], hhi.shape[1], dtype=torch.float64)
            for r0 in range(c0, min(B, c0 + CHUNK), 16):
                for a, h in terms:
                    accw = rnd(accw + a[r0:r0 + 16].T @ h[r0:r0 + 16])
            accb = rnd((zhi[c0:c0 + CHUNK] + zlo[c0:c0 + CHUNK]).sum(0))
            tot_w = accw if tot_w is None else rnd(tot_w + accw)
            tot_b = accb if tot_b is None else rnd(tot_b + accb)
        out[l] = (tot_w * 2.0 ** -s[l], tot_b * 2.0 ** -s[l])
        if l == 0:
            break
        whi, wlo = split(params[l][0])
        K = whi.shape[0]
        acc = torch.zeros(B, whi.shape[1], dtype=torch.float64)
        for k0 in range(0, K, 16):
            for a, w in ((zhi, whi), (zhi, wlo), (zlo, whi)):
                acc = rnd(acc + a[:, k0:k0 + 16] @ w[k0:k0 + 16])
        mh, ml = split(Hs[l])
        zsc = torch.where((mh != 0) | (ml != 0), acc.float() * 2.0 ** (s[l - 1] - s[l]), torch.zeros(()))
    return out


@pytest.mark.parametrize("rz", [False, True])
def test_simulated_accumulator_within_emulation_bound(rz):
    """The f32 accumulators restated (to nearest and toward zero) stay within half the emulation bound."""
    for i, shape in enumerate(CPU_SHAPES[:4]):
        pol, x, up = _case(i, shape, mean_loss=i % 2 == 0)
        ps = net_params(pol)
        Hs, zs = forward_emul(ps, x)
        em, s = backward_emul(ps, Hs, up)
        sim = _simulated_backward(ps, Hs, up, s, rz)
        be = backward_bounds(ps, x, Hs, zs, up, s)
        check_grads(sim, em, {l: (0.5 * be[l][0], 0.5 * be[l][1]) for l in be}, tag=str(i))


def _rejected(m, em, be):
    worst = 0.0
    for l in em:
        for j in (0, 1):
            worst = max(worst, float(((m[l][j] - em[l][j]).abs() / be[l][j]).max()))
    return worst


@pytest.mark.parametrize("mutation", ["hilo_one_kblock", "no_scale", "bias_chunk", "mask_layer"])
def test_emulation_bound_rejects_mutations(mutation):
    """Each mutated backward models a subtle kernel bug; the emulation bound must reject it (some gradient entry beyond its bound)."""
    if mutation == "no_scale":
        # N = 524 288 rows with a mean loss: the unscaled head gradient (~1e-6) lands in the f16 subnormal range
        pol = make_policy(32, 4, 64, (64,), seed=7)
        B = 524288
        x = random_dense(np.random.Generator(np.random.PCG64(13)), B, 32, 0.5).double()
        up = torch.randn(B, 5, generator=torch.Generator().manual_seed(3)) / B
    else:
        # 64 -> 128 -> 128 -> 8 + value (equal hidden widths: the wrong layer's mask has the right shape); 3 chunks of rows, or (a dropped
        # product of one K block, ~2^-12 of that block's partial sums) 16 rows: one issue per product, where the wgrad bound is tight
        pol = make_policy(64, 8, 128, (128,), seed=5)
        B = 16 if mutation == "hilo_one_kblock" else 3000
        x = random_dense(np.random.Generator(np.random.PCG64(12)), B, 64, 0.5).double()
        up = torch.randn(B, 9, generator=torch.Generator().manual_seed(4)) / B
    ps = net_params(pol)
    Hs, zs = forward_emul(ps, x)
    em, s = backward_emul(ps, Hs, up)
    be = backward_bounds(ps, x, Hs, zs, up, s)
    kw = {"hilo_one_kblock": dict(drop_hilo=(1, 1)), "no_scale": dict(no_scale=True), "bias_chunk": dict(skip_bias_chunk=1),
          "mask_layer": dict(wrong_mask=True)}[mutation]
    m, _ = backward_emul(ps, Hs, up, **kw)
    assert _rejected(m, em, be) > 1.0, mutation


# ----------------------------------------------------------------------------------------------- GPU
def _tc(pol, max_batch):
    from qiskit_gym_b200.policy import TensorCorePolicy
    return TensorCorePolicy(pol, max_batch=max_batch, device=0, with_value=True, training=True)


def _run(tcp, pol, bits, dl, dv):
    """forward_train + backward with upstream (dl, dv): {l: (dW, db)} read from .grad (zeroed first), and the forward's outputs."""
    from qiskit_gym_b200.policy import action_layers, simple_value_head
    pol.zero_grad(set_to_none=True)
    lg, v = tcp.forward_train(pol, bits)
    torch.autograd.backward([lg, v], [dl, dv.reshape(-1, 1)])
    layers = action_layers(pol)
    head = simple_value_head(pol)
    out = {}
    for l, lin in enumerate(layers):
        gW, gb = lin.weight.grad, lin.bias.grad
        if l == len(layers) - 1:
            gW = torch.cat([gW, head.weight.grad.reshape(1, -1)])
            gb = torch.cat([gb, head.bias.grad.reshape(1)])
        out[l] = (gW.clone(), gb.clone())
    return out, lg.detach(), v.detach()


def _gpu_case(obs, A, emb, common, scale, B, seed, dens=0.4):
    from qiskit_gym_b200.policy import pack_obs_bits
    pol = make_policy(obs, A, emb, common, seed=seed, scale=scale).cuda()
    dense = random_dense(np.random.Generator(np.random.PCG64(100 + seed)), B, obs, dens)
    bits = pack_obs_bits(dense).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    up = torch.randn(B, A + 1, generator=g, device="cuda") / B
    return pol, dense.cuda().double(), bits, up


def _check_against_refs(pol, x, got, up, tag):
    ps = [(W.cuda(), b.cuda()) for W, b in net_params(pol)]
    Hs, zs = forward_emul(ps, x)
    em, s = backward_emul(ps, Hs, up)
    check_grads(got, em, backward_bounds(ps, x, Hs, zs, up, s), tag=tag + " emulation")
    ref = module_grads(pol, x, up[:, :-1], up[:, -1])
    check_grads(got, ref, backward_bounds(ps, x, Hs, zs, up, s, module=True), tag=tag + " module")


GPU_SHAPES = [  # obs, A, emb, common, scale, B
    (256, 72, 512, (256,), 1.0, 129),           # the C3 policy
    (256, 72, 512, (256,), 1e-2, 127),
    (256, 72, 512, (256,), 30.0, 1),
    (64, 8, 128, (64,), 1.0, 300),              # two hidden widths that are not multiples of 128
    (9, 1, 64, (), 1.0, 200),                   # 2 layers, one action, the smallest observation
    (729, 127, 256, (128, 64), 1.0, 257),       # 4 layers, 127 actions, the largest observation
    (25, 8, 4096, (64,), 1.0, 129),             # a 4096-wide layer
    (36, 27, 200, (100,), 30.0, 1000),
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", GPU_SHAPES, ids=lambda s: "x".join(map(str, s[:4])) + f"_s{s[4]}_B{s[5]}")
def test_backward_envelope(shape):
    obs, A, emb, common, scale, B = shape
    pol, x, bits, up = _gpu_case(obs, A, emb, common, scale, B, seed=B % 97)
    tcp = _tc(pol, B)
    got, _, _ = _run(tcp, pol, bits, up[:, :A].contiguous(), up[:, A].contiguous())
    _check_against_refs(pol, x, got, up, str(shape))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [65536 + 77, 524288 + 77])
def test_backward_collector_batches(B):
    """The C3 policy at collector batch sizes (several chunks per split-K reduction); the upstream gradient of a mean loss."""
    pol, x, bits, up = _gpu_case(256, 72, 512, (256,), 1.0, B, seed=3, dens=0.3)
    tcp = _tc(pol, B)
    got, _, _ = _run(tcp, pol, bits, up[:, :72].contiguous(), up[:, 72].contiguous())
    _check_against_refs(pol, x, got, up, f"B={B}")


@pytest.mark.gpu
def test_backward_ppo_loss():
    """The real PPO loss (ppo.PPO.update's statement) on the forward_train outputs: its upstream gradient, captured, against both references."""
    B, A = 3000, 72
    pol, x, bits, _ = _gpu_case(256, A, 512, (256,), 1.0, B, seed=5)
    tcp = _tc(pol, B)
    g = torch.Generator(device="cuda").manual_seed(9)
    act = torch.randint(0, A, (B,), generator=g, device="cuda")
    logp_old = torch.log(torch.full((B,), 1.0 / A, device="cuda")) + 0.1 * torch.randn(B, generator=g, device="cuda")
    adv = torch.randn(B, generator=g, device="cuda")
    ret = torch.randn(B, generator=g, device="cuda")
    pol.zero_grad(set_to_none=True)
    logits, value = tcp.forward_train(pol, bits)
    caught = {}
    logits.register_hook(lambda gr: caught.__setitem__("dl", gr.clone()))
    value.register_hook(lambda gr: caught.__setitem__("dv", gr.clone()))
    logp_all = torch.log_softmax(logits.float(), dim=-1)
    logp = logp_all.gather(1, act[:, None]).squeeze(1)
    ratio = torch.exp(logp - logp_old)
    pi_loss = -torch.min(ratio * adv, torch.clamp(ratio, 0.9, 1.1) * adv).mean()
    v_loss = torch.nn.functional.mse_loss(value.float().reshape(-1), ret)
    entropy = -(logp_all.exp() * logp_all).sum(-1).mean()
    (pi_loss + 0.8 * v_loss - 0.01 * entropy).backward()
    up = torch.cat([caught["dl"], caught["dv"].reshape(B, 1)], 1)
    from qiskit_gym_b200.policy import action_layers, simple_value_head
    layers = action_layers(pol)
    got = {l: (lin.weight.grad, lin.bias.grad) for l, lin in enumerate(layers)}
    head = simple_value_head(pol)
    got[len(layers) - 1] = (torch.cat([got[len(layers) - 1][0], head.weight.grad]), torch.cat([got[len(layers) - 1][1], head.bias.grad]))
    _check_against_refs(pol, x, got, up, "ppo loss")


@pytest.mark.gpu
def test_backward_reproducible_and_independent_of_capacity_and_stale_rows():
    """Bit-identical gradients across repeated calls, across handles of different capacity, and after a larger batch left other values in
    every buffer past the batch (acts, dZ images, partials)."""
    B = 3 * 1024 + 77
    pol, x, bits, up = _gpu_case(256, 72, 512, (256,), 1.0, B, seed=8)
    dl, dv = up[:, :72].contiguous(), up[:, 72].contiguous()
    small = _tc(pol, B)
    g1, lg1, v1 = _run(small, pol, bits, dl, dv)
    g2, _, _ = _run(small, pol, bits, dl, dv)
    big = _tc(pol, 4 * B)
    Bb = 4 * B
    _, _, bits_b, up_b = _gpu_case(256, 72, 512, (256,), 1.0, Bb, seed=9)
    up_b = up_b * 1e4 + 7.0                       # sentinel-like values in every row of the larger batch
    _run(big, pol, bits_b, up_b[:, :72].contiguous(), up_b[:, 72].contiguous())
    g3, lg3, v3 = _run(big, pol, bits, dl, dv)
    for l in g1:
        for j in (0, 1):
            assert torch.equal(g1[l][j], g2[l][j]), (l, j)
            assert torch.equal(g1[l][j], g3[l][j]), (l, j)
    assert torch.equal(lg1, lg3) and torch.equal(v1, v3)


@pytest.mark.gpu
def test_forward_train_matches_forward_bits():
    """The training handle's logits and values are bit-identical to forward_bits of a handle in per-layer mode."""
    from qiskit_gym_b200.policy import TensorCorePolicy
    B = 1000
    pol, x, bits, up = _gpu_case(256, 72, 512, (256,), 1.0, B, seed=11)
    ref = TensorCorePolicy(pol, max_batch=B, device=0, with_value=True)
    ref.set_per_layer(True)
    lg = torch.empty(B, 72, device="cuda")
    v = torch.empty(B, device="cuda")
    ref.forward_bits(bits, logits=lg, values=v)
    tcp = _tc(pol, B)
    lg2, v2 = tcp.forward_train(pol, bits)
    assert torch.equal(lg, lg2) and torch.equal(v, v2.reshape(-1))


@pytest.mark.gpu
def test_forward_train_backward_syncs_nothing_and_refuses_stale_graph():
    B = 500
    pol, x, bits, up = _gpu_case(64, 8, 128, (64,), 1.0, B, seed=12)
    tcp = _tc(pol, B)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        lg, v = tcp.forward_train(pol, bits)
        torch.autograd.backward([lg, v], [up[:, :8].contiguous(), up[:, 8:].contiguous()])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    lg, v = tcp.forward_train(pol, bits)
    tcp.forward_train(pol, bits)                  # a newer forward on the same handle
    with pytest.raises(ValueError):
        (lg.sum() + v.sum()).backward()


def _ppo(update_precision, seed=3, **kw):
    from qiskit_gym_b200.ppo import PPO
    from qiskit_gym_b200.search import BasicPolicy
    from tests.helpers import config_table
    kind, n, gs, ckw = config_table()["C1_perm_grid3"]
    torch.manual_seed(0)
    pol = BasicPolicy([n, n], len(gs), embedding_size=128, common_layers=(64,))
    cfg = {"collecting": {"num_episodes": 600}, "training": {"num_epochs": 1}}
    return PPO(kind, n, gs, pol, cfg, device=0, seed=seed, matmul_precision="tensor_core", update_precision=update_precision,
               difficulty=3, **dict(ckw, add_perms=True), **kw)


@pytest.mark.gpu
def test_ppo_tensor_core_update_gradients_within_contract():
    """One update step on the same rollout, tensor-core update against the f32 update: the gradients the tensor-core backward wrote are
    within the contract of float64 autograd given the upstream gradient the loss produced; the f32 update's gradients are within the
    same bound plus what the forward's error moves the loss's gradient by (checked loosely, relative to the gradient's scale)."""
    from qiskit_gym_b200.collector import unpack_bits
    ppo = _ppo("tensor_core")
    ro = ppo.collector.collect_packed(ppo._episode_steps())
    ref = _ppo("f32")
    ref.policy.load_state_dict(ppo.policy.state_dict())
    grads = {}
    for name, tr in (("tc", ppo), ("f32", ref)):
        tr._step = lambda loss, tr=tr, name=name: (tr.opt.zero_grad(set_to_none=True), loss.backward(),
                                                   grads.__setitem__(name, [p.grad.clone() for p in tr.policy.parameters()]))
        tr.update(ro)
    for a, b in zip(grads["tc"], grads["f32"]):
        scale = float(b.abs().max()) + 1e-30
        assert float((a - b).abs().max()) <= 1e-3 * scale, float((a - b).abs().max()) / scale
    # the contract itself, on the tensor-core update's own upstream gradient
    idx = ro.valid.reshape(-1).nonzero(as_tuple=False).squeeze(1)
    bits = ro.obs_bits.reshape(-1, ro.obs_bits.shape[-1])[idx]
    tcp = ppo._train_policy(bits.shape[0])
    B = bits.shape[0]
    g = torch.Generator(device="cuda").manual_seed(1)
    up = torch.randn(B, ppo.env.num_actions() + 1, generator=g, device="cuda") / B
    A = ppo.env.num_actions()
    got, _, _ = _run(tcp, ppo.policy, bits, up[:, :A].contiguous(), up[:, A].contiguous())
    x = unpack_bits(bits, ro.obs_size).double()
    _check_against_refs(ppo.policy, x, got, up, "ppo rollout")


@pytest.mark.gpu
def test_ppo_update_precision_refusals():
    from qiskit_gym_b200.ppo import PPO
    from qiskit_gym_b200.search import BasicPolicy
    from tests.helpers import config_table
    kind, n, gs, ckw = config_table()["C1_perm_grid3"]
    pol = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(64,))
    with pytest.raises(ValueError):
        PPO(kind, n, gs, pol, {"collecting": {"num_episodes": 64}}, device=0, matmul_precision="f32", update_precision="tensor_core", **ckw)
    with pytest.raises(ValueError):
        PPO(kind, n, gs, pol, {"collecting": {"num_episodes": 64}}, device=0, update_precision="bf16", **ckw)
    deep = BasicPolicy([n, n], len(gs), embedding_size=64, common_layers=(64,), value_layers=(32,))
    with pytest.raises(NotImplementedError):
        PPO(kind, n, gs, deep, {"collecting": {"num_episodes": 64}}, device=0, matmul_precision="tensor_core", update_precision="tensor_core", **ckw)


def test_alphazero_refuses_tensor_core_update():
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2)], difficulty=1)
    rls = RLSynthesis(env, {}, {"embedding_size": 16, "common_layers": [16]}, device=None)
    rls.algorithm_cls = "twisterl.rl.AZ"
    with pytest.raises(NotImplementedError):
        rls.learn(num_iterations=1, update_precision="tensor_core")


@pytest.mark.gpu
def test_ppo_tensor_core_update_learns_permutation_line4(tmp_path):
    """test_collector_packed.py::test_ppo_tensor_core_learns_permutation_line4 with the update on the tensor cores as well."""
    from qiskit_gym_b200.rl import RLSynthesis
    from qiskit_gym_b200.specs import SynthSpec

    torch.manual_seed(0)
    env = SynthSpec.from_coupling_map("PermutationEnv", [(0, 1), (1, 2), (2, 3)], difficulty=1, depth_slope=2, max_depth=32)
    cfg = {"collecting": {"num_episodes": 512}, "training": {"num_epochs": 4, "ent_coef": 0.01}, "optimizer": {"lr": 2e-3},
           "learning": {"diff_threshold": 0.85, "diff_max": 8, "diff_metric": "ppo_deterministic"},
           "evals": {"ppo_deterministic": {"num_episodes": 128}}, "logging": {"log_freq": 1, "checkpoint_freq": 20}}
    rls = RLSynthesis(env, cfg, {"embedding_size": 64, "common_layers": [64]}, device=0)
    targets = [list(np.random.Generator(np.random.PCG64(s)).permutation(4)) for s in range(24)]
    targets = [t for t in targets if t != [0, 1, 2, 3]]
    before = sum(rls.synth(t, deterministic=True, num_searches=1) is not None for t in targets)
    hist = rls.learn(initial_difficulty=1, num_iterations=40, tb_path=str(tmp_path), matmul_precision="tensor_core",
                     update_precision="tensor_core")
    assert len(hist) == 40 and hist[-1]["difficulty"] >= 4, [(h["difficulty"], round(h["eval/ppo_deterministic"], 2)) for h in hist]
    after = sum(rls.synth(t, deterministic=True, num_searches=1) is not None for t in targets)
    assert after >= max(before + 5, int(0.8 * len(targets))), (before, after, len(targets))
