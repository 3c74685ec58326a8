"""Every launch of the fused training step, element by element against fp64, on the operands it actually read.

The step runs as production runs it: FusedTrainStep(graph=True) with the next batch prefetched on the background stream
and the gradient buffer cleared by Adam (keep_grads=False). For the last two steps of a run the test snapshots the
flat state before the step (a synchronisation, outside the replayed graph) and reads back what the step left: the
activation planes of the plan's workspace, mu / logvar / eps, the loss-ring slot, the new parameters, moments and
shadow planes. test_step_reference_cpu.step_reference then rebuilds each launch from its OWN stored inputs in fp64:

    F1 h1 | F2 mu, logvar, z | F3 h3 | F4 da4, loss, db4 | B4d da3, db3 | B3d + latent d_ml, db2 | B2d da1, db1
    | B4w..B1w dW4..dW1 | Adam m, v, p, shadows

Gradients are never read directly (the step clears them): they are checked through Adam's first moment,
m_new = m + (1 - beta1)(coef g - m), per element, so this is exactly the gradient the production route fed to Adam.

Bounds are per element (see step_reference): |out - ref| <= E + the rounding of the stored output. A per-element
bound can be loose when K is large, so every matrix is also cut into 128 x 128 tiles, and a tile whose RMS of
|out - ref| / bound exceeds TILE_FACTOR times the median tile of the same tensor is flagged: a missing k-block or a
wrong split range in one tile shows there even under the per-element bound. Failure messages name the tensor, the
tile (row block, column block) and the worst element.

Each case reaches one route of the step, and asserts it by the launch count of an eager step of the same shapes
(tile choices replayed from choose_tile in csrc/gemm_host.cu for 148 SMs):
    default dims, B = 8192      fused dgrad + weight-gradient launches in stages 0 and 2, two-stream stage 1,
                                split-K weight gradients (bf16 and fp32 mode)
    default dims, B = 4096      frames read in place (sample span), 128-wide head tiles
    default dims, 8192 -> 8155  the ragged batch of an epoch tail: the schedules belong to B = 8192, separate launches
    (256, 320, 64), B = 1 / 128 single-CTA tiles and no stage-1 split; 129: a pair tile with one valid row; 300
    (512, 768, 192), B = 1300   L % 128 != 0: head with 3 column blocks, ragged rows
    (1000, 300, 16), B = 200    padded plan: the true columns are checked, every padding element must stay zero
    default dims, clipped       max_grad_norm with coef < 1, cosine lr with warm-up, cyclical beta: one Adam launch
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import pytest
import torch

from test_step_reference_cpu import U23, U24, step_reference

pytestmark = pytest.mark.gpu

DEFAULT = (1024, 2048, 256)
LR, KL_BETA, HOP = 1e-4, 1e-4, 128
# Tile-RMS outlier factor, calibrated on an NVIDIA B200 at its 1000 W power limit: over every case below, the largest
# ratio of a tile's RMS |err| / bound to the median tile of the same tensor was 1.7.
TILE_FACTOR = 8.0
TILE = 128


@dataclass
class Case:
    dims: tuple
    precision: str
    batch: int
    first_batch: Optional[int] = None   # batch size of the first steps (schedule owner), None = batch
    in_place: bool = False              # consecutive frames read in place instead of a random gather
    fused: tuple = (False, False)       # stages 0 and 2 run as one fused dgrad + weight-gradient launch
    clip: Optional[float] = None
    schedule: dict = field(default_factory=dict)


CASES = {
    "default_gather_bf16": Case(DEFAULT, "bf16", 8192, fused=(True, True)),
    "default_gather_fp32": Case(DEFAULT, "fp32", 8192, fused=(True, True)),
    "default_in_place_4096": Case(DEFAULT, "bf16", 4096, in_place=True, fused=(True, True)),
    "default_ragged_8155_after_8192": Case(DEFAULT, "bf16", 8155, first_batch=8192),
    "small_b1": Case((256, 320, 64), "bf16", 1),
    "small_b128": Case((256, 320, 64), "bf16", 128),
    "small_b129": Case((256, 320, 64), "bf16", 129),
    "small_b300": Case((256, 320, 64), "bf16", 300),
    "l192_b1300": Case((512, 768, 192), "bf16", 1300),
    "padded_b200": Case((1000, 300, 16), "bf16", 200),
    "default_clip_cosine_cyclical": Case(DEFAULT, "bf16", 8192, fused=(True, True), clip=1e-4,
                                         schedule=dict(lr_schedule="cosine", warmup_steps=3, total_steps=20,
                                                       lr_min=1e-5, kl_anneal="cyclical", kl_beta_start=0.0,
                                                       kl_cycles=2, kl_cycle_ratio=0.9)),
}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _cdiv(a, b):
    return -(-a // b)


def reduce_split(M, N, K, sms):
    """(K_split, n_splits) of a reduce-add GEMM: gemm_prepare's split-K choice (csrc/gemm_host.cu)."""
    cg = 2 if M > 128 else 1
    block_n = 256 if N % 256 == 0 else 128
    tiles = _cdiv(M, 128 * cg) * _cdiv(N, block_n)
    slots = sms // cg
    kb = _cdiv(K, 64)
    best, splits, s = 0.0, 1, 1
    while s <= 8 and kb // s >= 8:
        units = tiles * s
        eff = units / (_cdiv(units, slots) * slots)
        if eff > best + 1e-9:
            best, splits = eff, s
        if eff >= 0.90:
            break
        s += 1
    splits = min(splits, kb)
    per = _cdiv(kb, splits)
    return per * 64, _cdiv(kb, per)


def expected_launches(case):
    """Kernels of one eager training step with a prefetched next batch (rvae_plan_train_step): next batch gather +
    its noise, F1..F4, stage 0, Adam(W4) in the background, stage 1 (latent dgrad, weight gradient, latent backward),
    stage 2, stage 3, the final Adam. A fused stage is one launch, a separate one two. Clipping: the four norm
    launches replace the background Adam and join the single Adam launch."""
    stages = sum(1 if f else 2 for f in case.fused)
    return (15 if case.clip is not None else 12) + stages


# ------------------------------------------------------------------------------------------------ the checker
def _val(p):
    return p[0] if p[1] is None else p[0] + p[1]


class Checker:
    """Per-element and tile-RMS checks; collects failures and the largest |err| / bound and tile ratio per tensor."""

    def __init__(self, label):
        self.label, self.failures, self.stats = label, [], {}

    def check(self, name, got, ref, bound):
        got, ref, bound = got.double(), ref.double(), bound.double()
        assert got.shape == ref.shape == bound.shape, (name, got.shape, ref.shape, bound.shape)
        g2, r2, b2 = (t.reshape(1, -1) if t.dim() == 1 else t for t in (got, ref, bound))
        err = (g2 - r2).abs()
        ratio = torch.where(b2 > 0, err / b2.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
        ratio = torch.where(torch.isnan(ratio) | torch.isnan(g2), torch.full_like(ratio, math.inf), ratio)
        worst = float(ratio.max())
        if worst > 1.0:
            i = int(ratio.argmax())
            r, c = divmod(i, ratio.shape[1])
            self.failures.append(f"{self.label} {name}: element ({r}, {c}) in tile ({r // TILE}, {c // TILE}): "
                                 f"got {float(g2[r, c]):.9g}, reference {float(r2[r, c]):.9g}, |err| "
                                 f"{float(err[r, c]):.3e} > bound {float(b2[r, c]):.3e} ({worst:.3g} x)")
        tile_max = self._tiles(name, ratio) if got.dim() == 2 else 0.0   # bias vectors: per element only
        prev = self.stats.get(name, (0.0, 0.0))
        self.stats[name] = (max(prev[0], worst), max(prev[1], tile_max))

    def _tiles(self, name, ratio):
        R, C = ratio.shape
        mb, nb = _cdiv(R, TILE), _cdiv(C, TILE)
        if mb * nb < 4:
            return 0.0
        pad = torch.zeros(mb * TILE, nb * TILE, dtype=torch.float64, device=ratio.device)
        cnt = torch.zeros_like(pad)
        pad[:R, :C] = ratio.clamp_max(1e30) ** 2
        cnt[:R, :C] = 1.0
        ms = pad.view(mb, TILE, nb, TILE).sum((1, 3)) / cnt.view(mb, TILE, nb, TILE).sum((1, 3))
        rms = ms.sqrt()
        med = float(rms.flatten().median())
        # a floor: residuals far below the bound everywhere (1e-3 of it) are not an outlier however they scatter
        thr = TILE_FACTOR * max(med, 1e-3)
        top = float(rms.max())
        if top > thr:
            i = int(rms.argmax())
            tr, tc = divmod(i, nb)
            blk = ratio[tr * TILE:(tr + 1) * TILE, tc * TILE:(tc + 1) * TILE]
            j = int(blk.argmax())
            er, ec = divmod(j, blk.shape[1])
            self.failures.append(f"{self.label} {name}: tile ({tr}, {tc}) RMS |err|/bound {top:.3e} is "
                                 f"{top / max(med, 1e-300):.1f} x the median tile ({med:.3e}); worst element "
                                 f"({tr * TILE + er}, {tc * TILE + ec}) at {float(blk.max()):.3e} of its bound")
        return top / max(med, 1e-3)


# ------------------------------------------------------------------------------------------------ one captured step
def _planes(p):
    hi, lo = p
    return hi.double(), (None if lo is None else lo.double())


def _frames(batch, S, Sp, precision):
    x = batch.materialize()
    if Sp != S:
        x = torch.nn.functional.pad(x, (0, Sp - S))
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16) if precision == "fp32" else None
    return hi.double(), (None if lo is None else lo.double())


def _blocks(flat, buf):
    """name -> the padded block of a flat buffer (W1 [Hp, Sp], W2 [2Lp, Hp], W3 [Hp, Lp], W4 [Sp, Hp], biases)."""
    from rawaudiovae_kelsey_b200.engine import param_layout_padded
    lay, Sp, Hp, Lp = param_layout_padded(flat.S, flat.H, flat.L)
    shapes = {"W1": (lay.w1, (Hp, Sp)), "W2": (lay.w2, (2 * Lp, Hp)), "W3": (lay.w3, (Hp, Lp)),
              "W4": (lay.w4, (Sp, Hp)), "b1": (lay.b1, (Hp,)), "b2": (lay.b2, (2 * Lp,)), "b3": (lay.b3, (Hp,)),
              "b4": (lay.b4, (Sp,))}
    return {k: buf[o:o + int(np.prod(s))].view(s) for k, (o, s) in shapes.items()}


def _snapshot(flat):
    torch.cuda.synchronize()
    s = {k: getattr(flat, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "shadow_hi")}
    s["shadow_lo"] = flat.shadow_lo.clone() if flat.shadow_lo is not None else None
    s["step"] = int(flat.step.item())
    return s


def _readback(plan, flat, loss_slot):
    torch.cuda.synchronize()
    lib = plan.lib
    act = {n: tuple(None if t is None else t.clone() for t in plan.activation(n))
           for n in ("h1", "z", "h3", "da4", "da3", "d_ml", "da1")}
    fn = {"eps": lib.rvae_plan_eps, "mu": lib.rvae_plan_mu, "lv": lib.rvae_plan_logvar}
    lat = {k: plan._rows(int(f(plan.handle)), flat.Lp, flat.Lp).clone() for k, f in fn.items()}
    after = {k: getattr(flat, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "shadow_hi", "grads")}
    after["shadow_lo"] = flat.shadow_lo.clone() if flat.shadow_lo is not None else None
    after["step"] = int(flat.step.item())
    return act, lat, after, float(loss_slot)


def check_step(case, model, step, plan, batch, before, act, lat, after, loss, grad_norm, sms, label):
    """Rebuild every launch of one step from its stored inputs and check every output. Returns the Checker."""
    from rawaudiovae_kelsey_b200.schedule import Schedule
    flat = model._flat
    S, H, L = case.dims
    Sp, Hp, Lp = flat.Sp, flat.Hp, flat.Lp
    B = plan.batch
    prec = case.precision
    ck = Checker(label)
    sched = step.schedule if step.schedule is not None else Schedule()
    k = before["step"]
    beta_k = float(np.float32(sched.beta_at(k, step.kl_beta)))
    x = _frames(batch, S, Sp, prec)
    pl = lambda buf: _blocks(flat, buf)  # noqa: E731
    sh_hi = pl(before["shadow_hi"])
    sh_lo = pl(before["shadow_lo"]) if before["shadow_lo"] is not None else None
    W = {n: (sh_hi[n].double(), None if sh_lo is None else sh_lo[n].double()) for n in ("W1", "W2", "W3", "W4")}
    bias = {n: pl(before["params"])[n].double() for n in ("b1", "b2", "b3", "b4")}
    a = {("dml" if n == "d_ml" else n): _planes(p) for n, p in act.items()}
    la = {n: t.double() for n, t in lat.items()}
    c = dict(c0=float(np.float32(2.0 / (B * S))), c_kl=float(np.float32(beta_k / (B * L))),
             kl_scale=-0.5 * beta_k / (B * L), inv_rec=1.0 / (B * S),
             # tanh.approx.f32 in bf16 mode (absolute error below 2^-10.9), tanhf (2 ulp) in fp32 mode; expf: 2 ulp
             tanh_abs=2.0 ** -10.5 if prec == "bf16" else 0.0, tanh_rel=0.0 if prec == "bf16" else 4 * U24,
             exp_rel=4 * U24,
             # a thread of the OUT / HEAD epilogue sums its row of every tile it owns; column sums: warp tree, four
             # warps, one atomic per row block (GEMM epilogues) or per block of the latent kernel (<= 4 per SM)
             loss_n=_cdiv(B, 128) * max(Sp, 2 * Lp), cs_n=_cdiv(B, 128) + 64 + 4 * sms,
             split={"B3d": reduce_split(B, Lp, Hp, sms), "B4w": reduce_split(Sp, Hp, B, sms),
                    "B3w": reduce_split(Hp, Lp, B, sms), "B2w": reduce_split(2 * Lp, Hp, B, sms),
                    "B1w": reduce_split(Hp, Sp, B, sms)})
    ref = step_reference(x, W, bias, a, la, c)

    # stored activations: bf16 (half an ulp: 2^-8 relative) or hi + lo (the residual's half ulp: 2^-16 relative)
    rnd = 2.0 ** -8 if prec == "bf16" else 2.0 ** -16
    for name in ("h1", "z", "h3", "da4", "da3", "dml", "da1"):
        r, e = ref[name]
        got = _val(a[name])
        ck.check(name, got, r, e + rnd * (r.abs() + e))
    for name in ("mu", "lv"):
        r, e = ref[name]
        ck.check(name, la[name], r, e)
    # padding: columns past the true dims hold exact zeros (activation planes, latents)
    for name, true_cols in (("h1", H), ("h3", H), ("da3", H), ("da1", H), ("z", L), ("da4", S)):
        for p in a[name]:
            if p is not None and p.shape[1] > true_cols:
                assert bool((p[:, true_cols:] == 0).all()), f"{label} {name}: non-zero padding columns"
    if Lp != L:
        for p in a["dml"]:
            if p is not None:
                assert bool((p[:, L:Lp] == 0).all() and (p[:, Lp + L:] == 0).all()), f"{label} d_ml padding"
        for n in ("mu", "lv"):
            assert bool((la[n][:, L:] == 0).all()), f"{label} {n}: non-zero padding columns"
    # the loss of this step in its ring slot
    r, e = ref["loss"]
    ck.check("loss", torch.tensor([loss]), r.reshape(1).cpu(), (e + 2 * U24 * r.abs()).reshape(1).cpu())

    # gradients -> flat layout, then Adam: m, v per element against the reference gradient
    g = torch.zeros(flat.total, dtype=torch.float64, device=flat.params.device)
    eg = torch.zeros_like(g)
    gb, eb = _blocks(flat, g), _blocks(flat, eg)
    for n, src in (("W1", "dW1"), ("W2", "dW2"), ("W3", "dW3"), ("W4", "dW4"), ("b1", "db1"), ("b2", "db2"),
                   ("b3", "db3"), ("b4", "db4")):
        gb[n].copy_(ref[src][0])
        eb[n].copy_(ref[src][1])
    opt_g = step.optimizer.param_groups[0]
    b1_, b2_ = opt_g["betas"]
    lr_k = sched.lr_at(k, opt_g["lr"])
    t = k + 1
    f32 = lambda v: float(np.float32(v))  # noqa: E731
    step_size, sqrt_bc2 = f32(lr_k / (1.0 - b1_ ** t)), f32(math.sqrt(1.0 - b2_ ** t))
    omb1, beta2, omb2, eps = f32(1.0 - b1_), f32(b2_), f32(1.0 - b2_), f32(opt_g["eps"])
    coef = 1.0
    if case.clip is not None:
        norm_k = float(grad_norm)
        coef = f32(min(1.0, case.clip / (norm_k + 1e-6)))
        assert coef < 1.0, f"{label}: clipping did not engage (norm {norm_k})"
        gn = float(g.norm())
        assert abs(norm_k - gn) <= float(eg.norm()) + 1e-6 * gn, (label, norm_k, gn)
    m0, v0 = before["exp_avg"].double(), before["exp_avg_sq"].double()
    cg = coef * g
    m_ref = m0 + omb1 * (cg - m0)
    e_m = omb1 * coef * eg + 3 * U24 * (m0.abs() + omb1 * (cg.abs() + (cg - m0).abs()) + m_ref.abs())
    v_ref = beta2 * v0 + omb2 * cg * cg
    e_v = omb2 * (2 * cg.abs() * coef * eg + (coef * eg) ** 2) + 4 * U24 * (beta2 * v0 + omb2 * cg * cg + v_ref)
    mb, mr, me = _blocks(flat, after["exp_avg"]), _blocks(flat, m_ref), _blocks(flat, e_m)
    vb, vr, ve = _blocks(flat, after["exp_avg_sq"]), _blocks(flat, v_ref), _blocks(flat, e_v)
    for n in mb:
        ck.check(f"m[{n}]", mb[n], mr[n], me[n])
        ck.check(f"v[{n}]", vb[n], vr[n], ve[n])
    # the parameters from the kernel's own moments, within a few ulps; shadows and the cleared gradient exactly
    m1, v1 = after["exp_avg"].double(), after["exp_avg_sq"].double()
    upd = step_size * (m1 / (v1.sqrt() / sqrt_bc2 + eps))
    p_ref = before["params"].double() - upd
    ck.check("p", after["params"], p_ref, U24 * p_ref.abs() + 8 * U24 * upd.abs())
    p1 = after["params"]
    hi = p1.to(torch.bfloat16)
    assert torch.equal(after["shadow_hi"], hi), f"{label}: shadow_hi != rn_bf16(p)"
    if after["shadow_lo"] is not None:
        assert torch.equal(after["shadow_lo"], (p1 - hi.float()).to(torch.bfloat16)), f"{label}: shadow_lo"
    assert int((after["grads"] != 0).sum()) == 0, f"{label}: the gradient buffer is not zero after the step"
    assert after["step"] == k + 1, (label, after["step"], k)
    # padding of the flat buffer stays exactly zero
    true = torch.zeros(flat.total, dtype=torch.bool, device=g.device)
    for name in flat.geometry:
        flat.view(true, name).fill_(True)
    for n in ("params", "exp_avg", "exp_avg_sq"):
        assert int((after[n][~true] != 0).sum()) == 0, f"{label}: non-zero padding in {n}"
    return ck, ref, c


# ------------------------------------------------------------------------------------------------ running a case
def _audio(dev, n_frames, S, seed=3):
    from oracle.rawvae_oracle import synth_wav
    rng = np.random.default_rng(seed)
    return torch.from_numpy(synth_wav(rng, (n_frames - 1) * HOP + S)).to(dev)


def run_case(name, dev, keep=False):
    """Run a case to steady graph replay, check its last two steps. keep=True also returns what the planted-defect
    tests need."""
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import VAE, FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.schedule import Schedule
    case = CASES[name]
    S, H, L = case.dims
    torch.manual_seed(0)
    model = VAE(S, H, L, precision=case.precision).to(dev)
    model.eps_seed = 5
    opt = Adam(model.parameters(), lr=LR)
    step = FusedTrainStep(model, opt, KL_BETA, graph=True, schedule=Schedule(**case.schedule),
                          max_grad_norm=case.clip)
    first = case.first_batch or case.batch
    n_frames = 3 * max(first, case.batch) + 64
    audio = _audio(dev, n_frames, S)
    gen = torch.Generator().manual_seed(21)
    sms = ops.num_sms(dev)

    def batch(size, i):
        if case.in_place:
            return FrameBatch(audio, size, HOP, S, first_frame=(i * 997) % (n_frames - size))
        return FrameBatch(audio, size, HOP, S, frame_idx=torch.randint(0, n_frames, (size,), generator=gen).to(dev))

    sizes = [first] * (3 if case.first_batch else 0)
    batches = [batch(s, i) for i, s in enumerate(sizes)]
    eager_launches = None
    i = 0
    checked = []
    while True:
        while len(batches) < i + 2:
            batches.append(batch(case.batch, len(batches)))
        cur, nxt = batches[i], batches[i + 1]
        final = cur.n_frames == case.batch and step.steady >= 2
        flat = model._ensure_flat()
        before = _snapshot(flat) if final else None
        st0, l0 = dict(step.stats), ops.launch_count(dev)
        slot = step(cur, next_data=nxt)
        if step.stats["eager"] > st0["eager"] and cur.n_frames == case.batch:
            eager_launches = ops.launch_count(dev) - l0
        if final:
            assert step.stats["replays"] == st0["replays"] + 1, (name, step.stats)
            plan = model._plan_for(case.batch)
            assert plan.batch == case.batch
            act, lat, after, loss = _readback(plan, flat, slot)
            gn = step.grad_norm.item() if case.clip is not None else None
            checked.append((cur, before, act, lat, after, loss, gn, plan))
            if len(checked) == 2:
                break
        i += 1
        assert i < 24, (name, step.stats)
    assert eager_launches == expected_launches(case), (name, eager_launches, expected_launches(case))
    results = []
    for j, (cur, before, act, lat, after, loss, gn, plan) in enumerate(checked):
        ck, ref, c = check_step(case, model, step, plan, cur, before, act, lat, after, loss, gn, sms,
                                f"{name} step {before['step']}")
        results.append((ck, ref, c, before, after, act, cur))
    return (model, step, results) if keep else [r[0] for r in results]


def _report(checkers):
    for ck in checkers:
        for n, (w, t) in sorted(ck.stats.items()):
            print(f"STAT {ck.label} {n} max|err|/E {w:.3e} max tile ratio {t:.2f}")


@pytest.mark.parametrize("name", list(CASES))
def test_step_every_launch_elementwise(name, dev):
    checkers = run_case(name, dev)
    _report(checkers)
    failures = [f for ck in checkers for f in ck.failures]
    assert not failures, "\n".join(failures[:40])


# ------------------------------------------------------------------------------------------------ the checker itself
@pytest.fixture(scope="module")
def small_step(dev):
    return run_case("small_b300", dev, keep=True)


@pytest.fixture(scope="module")
def default_step(dev):
    return run_case("default_gather_bf16", dev, keep=True)


@pytest.mark.parametrize("tensor", ["h1", "da3"])
def test_checker_flags_one_element_at_tile_corners(tensor, small_step):
    """One element of a copy of a real step output pushed to 4 E at tile corners (rows 127 / 128 / 255 / 256 and the
    last, ragged row 299; columns 63 / 64 / 255 / 256): the checker names it."""
    _, _, results = small_step
    ck0, ref, c, _, _, act, _ = results[-1]
    got = _val(_planes(act[tensor]))
    r, e = ref[tensor]
    bound = e + 2.0 ** -8 * (r.abs() + e)
    clean = Checker("clean")
    clean.check(tensor, got, r, bound)
    assert not clean.failures, clean.failures
    for row in (127, 128, 255, 256, got.shape[0] - 1):
        for col in (63, 64, 255, 256):
            bad = got.clone()
            sign = 1.0 if float(bad[row, col] - r[row, col]) >= 0 else -1.0
            bad[row, col] = r[row, col] + sign * 4.0 * max(float(bound[row, col]), 1e-30)
            ck = Checker("planted")
            ck.check(tensor, bad, r, bound)
            assert any(f"({row}, {col})" in f for f in ck.failures), (row, col, ck.failures)


def test_checker_flags_a_dw1_tile_without_its_last_k_block(default_step):
    """One 256 x 256 tile of dW1 replaced by its value without the last k-block (the last 64 frames of the batch),
    planted in a copy of the first moment the step wrote: the tile is flagged."""
    model, step, results = default_step
    ck0, ref, c, before, after, act, cur = results[-1]
    flat = model._flat
    x = _frames(cur, model.segment_length, flat.Sp, "bf16")
    da1 = _planes(act["da1"])
    r0, r1, c0_, c1 = 256, 512, 256, 512
    K = da1[0].shape[0]
    last = (K - 1) // 64 * 64
    miss = da1[0][last:, r0:r1].T @ x[0][last:, c0_:c1]
    omb1 = float(np.float32(1.0 - step.optimizer.param_groups[0]["betas"][0]))
    m_bad = _blocks(flat, after["exp_avg"].double().clone())["W1"]
    m_bad[r0:r1, c0_:c1] -= omb1 * miss
    # the reference m of W1, rebuilt as check_step does it (coef = 1: this case does not clip)
    g, e = ref["dW1"]
    m0 = _blocks(flat, before["exp_avg"].double())["W1"]
    m_ref = m0 + omb1 * (g - m0)
    e_m = omb1 * e + 3 * U24 * (m0.abs() + omb1 * (g.abs() + (g - m0).abs()) + m_ref.abs())
    clean = Checker("clean")
    clean.check("m[W1]", _blocks(flat, after["exp_avg"])["W1"], m_ref, e_m)
    assert not clean.failures, clean.failures
    ck = Checker("planted")
    ck.check("m[W1]", m_bad, m_ref, e_m)
    # 128 x 128 tiles (2..3, 2..3) cover the planted 256 x 256 tile
    assert any(f"tile ({tr}, {tc})" in f for f in ck.failures for tr in (2, 3) for tc in (2, 3)), ck.failures


@pytest.mark.parametrize("bias", ["db1", "db3", "db4"])
def test_checker_flags_a_bias_column_without_one_row_block(bias, small_step):
    """One column of a bias gradient with one 128-row block's contribution removed: flagged."""
    _, _, results = small_step
    _, ref, c, _, _, _, _ = results[-1]
    src = {"db1": "da1", "db3": "da3", "db4": "da4"}[bias]
    v = ref[src][0]
    r, e = ref[bias]
    col = int(v[128:256].abs().sum(0).argmax())
    bad = r.clone()
    bad[col] -= v[128:256, col].sum()
    ck = Checker("planted")
    ck.check(bias, bad, r, e)
    assert any(f"(0, {col})" in f for f in ck.failures), (col, ck.failures)
