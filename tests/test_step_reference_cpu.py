"""Layer-local fp64 reference of one fused training step, and its check against the pinned oracle (no GPU needed).

`step_reference` recomputes every launch of rvae_plan_train_step from the operands that launch read - the bf16 planes
the step left in the plan's workspace, the bf16 shadow weights and fp32 biases it ran with - so an error in one launch
never propagates into the reference of the next. Every product is evaluated as the kernel issues it: hi*hi, plus
hi*lo + lo*hi when the operands carry residual planes (fp32 mode). Beside each reference value it returns a bound E on
the deviation a correct kernel may show, before the rounding of the stored output:

    E = gamma * sum_k |a_k| |b_k|,  gamma = (K_split * passes + n_splits + 2) * 2^-23

(fp32 accumulation that need not round to nearest, split-K partials reduce-added in fp32), carried through the
epilogue functions with explicit derivative bounds, plus a few fp32 ulps per elementary operation. Column sums (bias
gradients) and the loss get the sum of their terms' E plus n * 2^-23 * sum |terms| for n sequential fp32 additions.

tests/test_gpu_step_elementwise.py feeds it what a real step read and checks what the step wrote; this module ties it
to oracle.forward / oracle.backward, which are pinned against the reference implementation."""
from __future__ import annotations

import math

import torch

from oracle import rawvae_oracle as O

U23 = 2.0 ** -23
U24 = 2.0 ** -24


def _val(p):
    """Value of a (hi, lo) pair of planes."""
    return p[0] if p[1] is None else p[0] + p[1]


def _t(p):
    return (p[0].T, None if p[1] is None else p[1].T)


def mm(a, b, k_split=None, n_splits=1):
    """(a @ b, E) for operand planes a = (hi, lo) [M, K] and b = (hi, lo) [K, N] in fp64 (bf16 values are exact
    there): hi*hi, plus lo*hi and hi*lo when the residual planes exist - the passes the kernel issues."""
    (ah, al), (bh, bl) = a, b
    val = ah @ bh
    passes = 1
    if al is not None:
        val = val + al @ bh
        passes += 1
    if bl is not None:
        val = val + ah @ bl
        passes += 1
    aa = ah.abs() if al is None else ah.abs() + al.abs()
    bb = bh.abs() if bl is None else bh.abs() + bl.abs()
    ks = ah.shape[1] if k_split is None else k_split
    gamma = (ks * passes + n_splits + 2) * U23
    return val, gamma * (aa @ bb)


def _colsum(v, e, n_add):
    """Column sums of v [rows, cols] with their bound: the terms' bounds plus n_add sequential fp32 additions."""
    return v.sum(0), e.sum(0) + n_add * U23 * v.abs().sum(0)


def step_reference(x, W, b, act, lat, c):
    """Reference values and bounds for every launch of one training step (all tensors fp64, the plan's padded dims).

    x   : (hi, lo) planes of the frames [B, S]                    (lo = None in bf16 mode)
    W   : W1 [H, S], W2 [2L, H] (fc21 rows, then fc22 rows), W3 [H, L], W4 [S, H]: (hi, lo) shadow planes
    b   : b1 [H], b2 [2L], b3 [H], b4 [S]: the fp32 master biases
    act : h1, z, h3, da4, da3, dml, da1: (hi, lo) planes the step stored
    lat : mu, lv, eps [B, L]: what the step stored (mu / logvar) and drew (eps)
    c   : c0 (= 2 / (B S)), c_kl (= beta / (B L)), kl_scale (= -beta / (2 B L)), inv_rec (= 1 / (B S)),
          tanh_abs / tanh_rel (error of the kernel's tanh), exp_rel (of its expf), loss_n / cs_n (sequential fp32
          additions of the loss sums / of a column sum), split: GEMM name -> (K_split, n_splits) of the split-K GEMMs
    Returns name -> (reference, E). Weight and bias gradients are under dW1..dW4, db1..db4."""
    split = c.get("split", {})
    exp_rel = c["exp_rel"]
    out = {}
    relu = lambda t: t.clamp_min(0.0)  # noqa: E731

    # F1: h1 = relu(x W1^T + b1)
    acc, e = mm(x, _t(W["W1"]))
    pre = acc + b["b1"]
    out["h1"] = (relu(pre), e + U24 * pre.abs())

    # F2 (head): mu | logvar = h1 W2^T + b2; z = mu + eps exp(logvar / 2); the KL sum of the loss
    acc, e = mm(act["h1"], _t(W["W2"]))
    Lp = W["W2"][0].shape[0] // 2
    mu, lv = acc[:, :Lp] + b["b2"][:Lp], acc[:, Lp:] + b["b2"][Lp:]
    e_mu, e_lv = e[:, :Lp] + U24 * mu.abs(), e[:, Lp:] + U24 * lv.abs()
    eps = lat["eps"]
    sig = torch.exp(0.5 * lv)
    z = mu + eps * sig
    e_sig = sig * torch.expm1(0.5 * e_lv) + 2 * exp_rel * sig * torch.exp(0.5 * e_lv)
    out["mu"], out["lv"] = (mu, e_mu), (lv, e_lv)
    out["z"] = (z, e_mu + eps.abs() * e_sig + 2 * U24 * (z.abs() + (eps * sig).abs()))
    sig2 = sig * sig
    kl_terms = (1.0 + lv) - (mu * mu + sig2)
    e_sig2 = sig2 * torch.expm1(e_lv) + 3 * exp_rel * sig2 * torch.exp(e_lv)
    e_kl = e_lv + 2 * mu.abs() * e_mu + e_mu * e_mu + e_sig2 + 4 * U24 * ((1.0 + lv).abs() + mu * mu + sig2)
    kl_sum, e_kl_sum = kl_terms.sum(), e_kl.sum() + c["loss_n"] * U23 * kl_terms.abs().sum()

    # F3: h3 = relu(z W3^T + b3)
    acc, e = mm(act["z"], _t(W["W3"]))
    pre = acc + b["b3"]
    out["h3"] = (relu(pre), e + U24 * pre.abs())

    # F4 (out): t = tanh(h3 W4^T + b4); d = t - x; da4 = c0 d (1 - t^2); the MSE sum; db4 = column sums of da4
    acc, e = mm(act["h3"], _t(W["W4"]))
    a = acc + b["b4"]
    t = torch.tanh(a)
    e_t = e + U24 * a.abs() + c["tanh_abs"] + c["tanh_rel"] * t.abs()   # tanh is 1-Lipschitz
    d = t - _val(x)
    da4 = c["c0"] * d * (1.0 - t * t)
    # |d/dt (t - x)(1 - t^2)| = |1 - t^2 - 2t(t - x)| <= 5 for |t|, |x| <= 1
    e_da4 = c["c0"] * (5.0 * e_t + 3.0 * e_t * e_t) + 4 * U24 * da4.abs()
    out["da4"] = (da4, e_da4)
    out["db4"] = _colsum(da4, e_da4, c["cs_n"])
    rec = (d * d).sum()
    e_rec = (2 * d.abs() * e_t + e_t * e_t).sum() + c["loss_n"] * U23 * rec
    loss = c["inv_rec"] * rec + c["kl_scale"] * kl_sum
    out["loss"] = (loss, c["inv_rec"] * e_rec + abs(c["kl_scale"]) * e_kl_sum + 4 * U24 * abs(float(loss)))

    # B4d (dgrad + ReLU mask of the stored h3): da3 = (da4 W4) [h3 > 0]; db3
    acc, e = mm(act["da4"], W["W4"])
    m3 = (act["h3"][0] > 0).to(acc.dtype)
    out["da3"] = (acc * m3, e * m3)
    out["db3"] = _colsum(acc * m3, e * m3, c["cs_n"])

    # B3d (split-K dz = da3 W3) + latent backward: d_mu = dz + c mu, d_lv = dz eps sigma / 2 + c (sigma^2 - 1) / 2
    dz, e_dz = mm(act["da3"], W["W3"], *split.get("B3d", (None, 1)))
    mu_k, lv_k, ck = lat["mu"], lat["lv"], c["c_kl"]
    sig = torch.exp(0.5 * lv_k)
    dmu = dz + ck * mu_k
    g = 0.5 * dz * eps * sig
    dlv = g + 0.5 * ck * (sig * sig - 1.0)
    e_dmu = e_dz + 2 * U24 * (dz.abs() + (ck * mu_k).abs())
    e_dlv = (0.5 * eps.abs() * sig * e_dz + (4 * U24 + exp_rel) * g.abs()
             + 0.5 * abs(ck) * ((3 * U24 + 2 * exp_rel) * sig * sig + 2 * U24 * (sig * sig + 1.0)) + 2 * U24 * dlv.abs())
    dml, e_dml = torch.cat([dmu, dlv], 1), torch.cat([e_dmu, e_dlv], 1)
    out["dml"] = (dml, e_dml)
    out["db2"] = _colsum(dml, e_dml, c["cs_n"])

    # B2d (dgrad + ReLU mask of the stored h1): da1 = (d_ml W2) [h1 > 0]; db1
    acc, e = mm(act["dml"], W["W2"])
    m1 = (act["h1"][0] > 0).to(acc.dtype)
    out["da1"] = (acc * m1, e * m1)
    out["db1"] = _colsum(acc * m1, e * m1, c["cs_n"])

    # weight gradients: split-K reduce-adds over the batch
    out["dW4"] = mm(_t(act["da4"]), act["h3"], *split.get("B4w", (None, 1)))
    out["dW3"] = mm(_t(act["da3"]), act["z"], *split.get("B3w", (None, 1)))
    out["dW2"] = mm(_t(act["dml"]), act["h1"], *split.get("B2w", (None, 1)))
    out["dW1"] = mm(_t(act["da1"]), x, *split.get("B1w", (None, 1)))
    return out


# ------------------------------------------------------------------------------------------------ vs the oracle
def test_step_reference_reproduces_the_oracle():
    """Fed the oracle's own fp64 activations at the golden small dims (S, H, L, B = 128, 192, 64, 48; no residual
    planes, exact constants), the reference reproduces oracle.forward, loss_function and backward to 1e-12."""
    S, H, L, B, beta = 128, 192, 64, 48, 0.37
    p = {k: v.double() for k, v in O.init_params(S, H, L, seed=4).items()}
    gen = torch.Generator().manual_seed(5)
    x = (torch.rand(B, S, generator=gen, dtype=torch.float64) * 2 - 1)
    eps = torch.randn(B, L, generator=gen, dtype=torch.float64)
    a = O.forward(p, x, eps)
    g = O.backward(p, a, beta)
    ga = g["_act"]
    one = lambda t: (t, None)  # noqa: E731
    W = {"W1": one(p["fc1.weight"]), "W2": one(torch.cat([p["fc21.weight"], p["fc22.weight"]])),
         "W3": one(p["fc3.weight"]), "W4": one(p["fc4.weight"])}
    bias = {"b1": p["fc1.bias"], "b2": torch.cat([p["fc21.bias"], p["fc22.bias"]]), "b3": p["fc3.bias"],
            "b4": p["fc4.bias"]}
    act = {"h1": one(a["h1"]), "z": one(a["z"]), "h3": one(a["h3"]), "da4": one(ga["da4"]), "da3": one(ga["da3"]),
           "dml": one(torch.cat([ga["dmu"], ga["dlv"]], 1)), "da1": one(ga["da1"])}
    lat = {"mu": a["mu"], "lv": a["logvar"], "eps": eps}
    c = dict(c0=2.0 / (B * S), c_kl=beta / (B * L), kl_scale=-0.5 * beta / (B * L), inv_rec=1.0 / (B * S),
             tanh_abs=0.0, tanh_rel=0.0, exp_rel=0.0, loss_n=0, cs_n=0)
    ref = step_reference(one(x), W, bias, act, lat, c)

    expect = {"h1": a["h1"], "mu": a["mu"], "lv": a["logvar"], "z": a["z"], "h3": a["h3"], "da4": ga["da4"],
              "da3": ga["da3"], "dml": torch.cat([ga["dmu"], ga["dlv"]], 1), "da1": ga["da1"],
              "loss": O.loss_function(a["x_hat"], x, a["mu"], a["logvar"], beta, S),
              "dW1": g["fc1.weight"], "dW2": torch.cat([g["fc21.weight"], g["fc22.weight"]]), "dW3": g["fc3.weight"],
              "dW4": g["fc4.weight"], "db1": g["fc1.bias"], "db2": torch.cat([g["fc21.bias"], g["fc22.bias"]]),
              "db3": g["fc3.bias"], "db4": g["fc4.bias"]}
    assert set(expect) <= set(ref)
    for name, want in expect.items():
        got, e = ref[name]
        assert got.shape == want.shape, name
        err = float((got - want).abs().max()) / max(float(want.abs().max()), 1e-300)
        assert err < 1e-12, f"{name}: {err:.3e}"
        assert bool(torch.isfinite(torch.as_tensor(e)).all()) and bool((torch.as_tensor(e) >= 0).all()), name
