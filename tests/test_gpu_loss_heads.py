"""The fused loss heads of the training steps against fp64 references, at the logit gradient and at the training shape.

``TrainStep._head`` turns logits into (loss, logit gradient) by composing the kernels of csrc/losses.cu with the weights and
scales of each script; this file calls it directly on synthetic logits, so no network and no BatchNorm sums are involved and
the comparison can be tight.  It also pins the mean-teacher consistency kernels (UAMT / USTM), rot90 and its use in
``USTMStep._body``, the run-to-run determinism of every ticket reduction, and the nearest resize of the UNet_DS heads.

Reference: the oracle's formulas (wsl_oracle) in fp64 on the device with autograd to the logits.  Discontinuous parts -- TV's
pooling argmin/argmax, the sign of |dp| in Mumford-Shah's gradientLoss2d, the mixed pseudo-label argmax, the UAMT mask -- come
from torch fp32 on CUDA applied to the head's own fp32 probabilities, so ties break as they do when the reference trains.

Tolerances, fp32 mode:
  loss and each regulariser's buffer value               1e-5 relative to fp64
  per-sample / per-class intermediates (CRF kernel mass, MS centroids, Dice I/Y/Z sums, variance mean/std)
                                                         1e-5 relative, with a floor of 1e-5 x the largest entry of the same
                                                         quantity (saturated logits leave ~1e-50 in fp64 where fp32 has 0);
                                                         1e-4 for the variance statistics of near-uniform probabilities, whose
                                                         inter-class std is a difference of nearly equal class means summed in
                                                         fp32 block partials (measured 5.4e-5)
  entropy of saturated probabilities                     against torch fp32 on the head's probabilities: p + 1e-6 at p = 1 is
                                                         1 + 8 ulp in fp32, 4.6 % off 1e-6, in the kernel and in the reference's
                                                         own fp32 arithmetic alike
  dlogits                                                1e-5 x max|g_ref|, elementwise; 1.2e-4 for near-uniform probabilities
                                                         without labels, where the regulariser sets max|g_ref|: the softmax
                                                         Jacobian's g_c - sum_k g_k p_k cancels ~20x in fp32 (CRF: 2.6e-5) and
                                                         the variance term inherits its inter-class std's error (5.7e-5)
  dlogits on unlabelled pixels (pCE adds exactly 0)      rel-L2 1e-4 against the regulariser's own fp64 gradient (4e-4 for the
                                                         variance term of near-uniform probabilities, measured 1.7e-4); where
                                                         that gradient is below fp32's range (saturated softmax) it must be 0
  TV probability gradient                                same support as torch's (residues of torch's own fp32 sums below half
                                                         a unit g = 1e-2 / numel count as 0), values 1e-6 relative; sample 0
                                                         gets none
  pseudo labels                                          bit-identical to torch.argmax of the fp32 mix
bf16 / fp16 modes: channels 0-3 of the NHWC-16 gradient are exactly round-to-nearest(S x fp32-mode dlogits) (S, the fp16 loss
scale, is a power of two; 1 in bf16), channels 4-15 are 0; fp16 at 64x256x256 has no inf and flushes to zero at most
FP16_FLUSH_MAX of the nonzero elements (measured on a B200).
Consistency kernels: sum / count / loss 1e-5 relative, mask identical more than 1e-5 away from the threshold, dlogits rel-L2 1e-5.
rot90, nearest resize, ticket reductions: bit-exact.

Labels with values >= 5 that are not ignore_index are skipped by the kernels like ignored pixels (torch's cross_entropy would
raise); with no labelled pixel at all the loss is NaN, as torch gives, and the logit gradient is the regulariser's alone.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import wsl_oracle as O
from _gpu_util import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"

if torch.cuda.is_available():
    from wsl4mis_b200._lib import call, workspace
    from wsl4mis_b200.engine import VARIANTS, TrainStep, USTMStep
    from wsl4mis_b200.networks.unet import UNet, UNet_CCT
else:
    VARIANTS = ()

FULL = (64, 256, 256)          # per-GPU batch of BASELINE config 2
VAR_ITER = 27000               # pce_variance ramp: 0.1 * sigmoid_rampup(180, 200) = 0.095
DMPLS_BETA = 0.3               # not a dyadic number: float(beta) and float(1 - beta) both round
# largest fraction of the nonzero fp32-mode logit-gradient elements (x S) that fp16 flushes to zero at 64x256x256, 'trained'
# logits, 3 % scribbles; measured on a B200 (1000 W) in the comment, bounded with ~2x headroom
FP16_FLUSH_MAX = {
    "pce": 1e-6,             # 0
    "pce_gatedcrf": 2e-6,    # 5.4e-7
    "pce_ms": 2e-6,          # 8.9e-7
    "pce_tv": 3e-2,          # 1.45e-2: TV routes g = 1e-2 / numel ~ 6e-10 per pixel, under p(1 - p) often below fp16's range
    "dmpls": 1.5e-4,         # 3.6e-5 (main head), 6.3e-5 (aux head)
    "pce_entropy": 6e-6,     # 2.6e-6
    "pce_variance": 2.5e-3,  # 1.3e-3: the variance term's logit gradients are ~1e-13 where the class variance is flat
}

_STEPS = {}


def _step(variant, precision):
    key = (variant, precision)
    if key not in _STEPS:
        torch.manual_seed(0)
        m = (UNet_CCT if variant == "dmpls" else UNet)(1, 4).to(DEV).set_precision(precision)
        st = TrainStep(m, variant, graph=False)
        st.ex.dev = torch.device(DEV)        # the executor learns its device in forward(); the head is called here without one
        _STEPS[key] = st
    st = _STEPS[key]
    st.iter_num = VAR_ITER
    st.beta_dev.copy_(torch.tensor([DMPLS_BETA, 1.0 - DMPLS_BETA], dtype=torch.float32))
    return st


def _logits(regime, N, H, W, seed, heads):
    """init: N(0, 0.05^2), near-uniform probabilities; trained: smooth class blobs at scale 3 (edges for CRF / TV);
    saturated: +-60, beyond fp32's exp range, so the fp32 probabilities are exactly 0 and 1 (at +-40 the losers would still hold
    e^-80 ~ 1.8e-35, a normal fp32 number)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = []
    for _ in range(heads):
        if regime == "init":
            x = 0.05 * torch.randn(N, 4, H, W, generator=g, device=DEV)
        else:
            z = torch.randn(N, 4, H // 16 + 2, W // 16 + 2, generator=g, device=DEV)
            z = F.interpolate(z, size=(H, W), mode="bilinear", align_corners=True)
            if regime == "trained":
                x = 3.0 * z + 0.3 * torch.randn(N, 4, H, W, generator=g, device=DEV)
            else:
                win = F.one_hot(z.argmax(1), 4).permute(0, 3, 1, 2).bool()
                x = torch.where(win, 60.0, -60.0)
        out.append(x.contiguous())
    return out


def _batch(labels, N, H, W, seed):
    """image U[0,1) and labels: 'scribble' (3 %), 'dense', 'none' (no labelled pixel), 'high' (scribbles plus 2 % of values in
    5..255, which are not ignore_index)"""
    image, lab = O.synth_batch(N, H, W, seed=seed, frac=0.03, dense=(labels == "dense"))
    if labels == "none":
        lab.fill_(4)
    elif labels == "high":
        g = torch.Generator().manual_seed(seed + 1)
        m = torch.rand(lab.shape, generator=g) < 0.02
        lab[m] = torch.randint(5, 256, (int(m.sum()),), generator=g, dtype=torch.uint8)
    return image.to(DEV), lab.to(DEV)


def _close(got, ref, rtol=1e-5):
    """max violation of |got - ref| <= rtol * max(|ref|, max|ref| * rtol-floor) as a ratio (<= 1 passes)"""
    got, ref = got.double().flatten(), ref.to(got.device).double().flatten()
    floor = ref.abs().max().clamp_min(1e-300)
    return ((got - ref).abs() / (rtol * torch.maximum(ref.abs(), 1e-5 * floor))).max().item()


def _rel(a, b):
    return abs(a - b) / abs(b) if b != 0 else abs(a)


def _grad(fn, x):
    """(value, d value / d x) of a scalar function of a fresh fp64 leaf copied from x"""
    leaf = x.detach().double().clone().requires_grad_(True)
    v = fn(leaf)
    (g,) = torch.autograd.grad(v, leaf)
    return v.item(), g


def _buf(step, name, shape, dt=torch.float32):
    return step.ex.buf("t", "head." + name, shape, dt)


# ------------------------------------------------------------------------------------------------------------------------
# fp64 references of the seven step bodies
# ------------------------------------------------------------------------------------------------------------------------
def _reference(variant, step, logits, image, label, regime):
    """-> dict(loss, g_ce [per head], g_reg [per head or None], checks {name: (got, ref)}, w)"""
    N, C, H, W = logits[0].shape
    lab_ref = torch.where(label < 4, label, torch.full_like(label, 4)).long()
    labelled = bool((lab_ref != 4).any())
    img64 = image.double()
    heads = 2 if variant == "dmpls" else 1
    w_ce = 0.5 if variant == "dmpls" else 1.0
    r = {"g_ce": [], "g_reg": [None] * heads, "checks": {}, "loss": 0.0}
    for h in range(heads):
        if labelled:
            ce, g = _grad(lambda x: w_ce * O.pce_loss(x, lab_ref), logits[h])
        else:
            ce, g = float("nan"), torch.zeros_like(logits[h], dtype=torch.float64)
        r["loss"] += ce
        r["g_ce"].append(g)
    probs = [_buf(step, f"probs{h}", (N, C, H, W)) for h in range(heads)]
    r["checks"]["probs"] = (probs[0], torch.softmax(logits[0].double(), 1))

    if variant == "pce_gatedcrf":
        val, ksum, g = 0.0, 0.0, torch.zeros_like(logits[0], dtype=torch.float64)
        for s in range(0, N, 8):                # sample-separable: chunks bound the fp64 graph's memory
            e = min(N, s + 8)
            frac = (e - s) / N
            v, g[s:e] = _grad(lambda x: 0.1 * frac * O.gated_crf_loss(torch.softmax(x, 1), img64[s:e]), logits[0][s:e])
            val += v / 0.1
            with torch.no_grad():                # kernels.sum(): the loss of an all-zero prediction times N*H*W
                ksum += O.gated_crf_loss(torch.zeros(e - s, C, H, W, dtype=torch.float64, device=DEV), img64[s:e]).item() * (e - s) * H * W
        crf = _buf(step, "crf", (2,))
        r["checks"]["crf"] = (crf[0:1], torch.tensor([val]))
        r["checks"]["crf.ksum"] = (crf[1:2], torch.tensor([ksum]))
        r["loss"] += 0.1 * val
        r["g_reg"][0] = g
    elif variant == "pce_ms":
        q = probs[0]
        sh, sw = torch.sign(q[:, :, 1:] - q[:, :, :-1]).double(), torch.sign(q[..., 1:] - q[..., :-1]).double()

        def ms(x):
            p = torch.softmax(x, 1)
            dh, dw = p[:, :, 1:] - p[:, :, :-1], p[..., 1:] - p[..., :-1]
            # |dp| keeps its fp64 value but takes its derivative from the sign of the head's fp32 difference (ties -> 0, as torch)
            fix = (sh * dh - dh.abs()).sum() + (sw * dw - dw.abs()).sum()
            return 1e-6 * (O.mumford_shah_loss(img64, p) + fix)
        v, g = _grad(ms, logits[0])
        with torch.no_grad():
            p = torch.softmax(logits[0].double(), 1)
            cent = (p * img64).sum((2, 3)) / img64.sum((2, 3))
        r["checks"]["ms"] = (_buf(step, "ms", (1,)), torch.tensor([v / 1e-6]))
        r["checks"]["cent"] = (_buf(step, "cent", (N * C,)), cent.flatten())
        r["loss"] += v
        r["g_reg"][0] = g
    elif variant == "pce_tv":
        gp = _buf(step, "gprobs0", (N, C, H, W))
        if N > 1:
            pr = probs[0].detach().clone().requires_grad_(True)
            (gtv,) = torch.autograd.grad(1e-2 * O.tv_loss(pr[1:]), pr)     # torch fp32 on CUDA: its argmin / argmax ties
            r["tv_gprobs"] = (gp, gtv)
            gtv = gtv.double()
            with torch.no_grad():
                tv = O.tv_loss(torch.softmax(logits[0].double(), 1)[1:]).item()
            _, g = _grad(lambda x: (torch.softmax(x, 1) * gtv).sum(), logits[0])
            r["checks"]["tv"] = (_buf(step, "tv", (1,)), torch.tensor([tv]))
            r["loss"] += 1e-2 * tv
            r["g_reg"][0] = g
        else:                                   # tv_loss(outputs_soft[1:]) of one image is a mean over nothing: no TV term
            r["tv_gprobs"] = (gp, torch.zeros_like(gp))
    elif variant == "pce_entropy":
        v, g = _grad(lambda x: 0.1 * O.entropy_loss(torch.softmax(x, 1), 4), logits[0])
        if regime == "saturated":               # see the module docstring: the value is torch's fp32 arithmetic, not fp64's
            v32 = O.entropy_loss(probs[0], 4).item()
            r["checks"]["ent"] = (_buf(step, "ent", (1,)), torch.tensor([v32]))
            r["loss"] += 0.1 * v32 - v            # the loss check then compares like with like as well
        else:
            r["checks"]["ent"] = (_buf(step, "ent", (1,)), torch.tensor([v / 0.1]))
        r["loss"] += v
        r["g_reg"][0] = g
    elif variant == "pce_variance":
        w = 0.1 * O.sigmoid_rampup(step.iter_num // 150, 200.0)
        v, g = _grad(lambda x: w * O.class_variance_loss(torch.softmax(x, 1), img64), logits[0])
        with torch.no_grad():
            vv = img64 * torch.softmax(logits[0].double(), 1)
            mean, sd = vv.mean((2, 3)), vv.std((2, 3))
            mbar, sdn = mean.mean(1), mean.std(1)
            stats = torch.cat([torch.stack([mean, sd], -1).flatten(), torch.stack([mbar, sdn], -1).flatten()])
            inter, intra = sdn.mean().item(), sd.mean().item()
        out = _buf(step, "var", (3,))
        r["checks"]["var"] = (out, torch.tensor([inter - intra, inter, intra]))
        r["checks"]["varstats"] = (_buf(step, "varstats", (N * C * 2 + N * 2,)), stats)
        r["loss"] += v
        r["g_reg"][0] = g
        r["w"] = w
    elif variant == "dmpls":
        pseudo = _buf(step, "pseudo", (N, H, W), torch.uint8)
        ref_pseudo = O.mix_pseudo_label(probs[0], probs[1], DMPLS_BETA).to(torch.uint8)   # fp32 on CUDA, torch's rounding
        r["pseudo"] = (pseudo, ref_pseudo)
        t = F.one_hot(ref_pseudo.long(), 4).permute(0, 3, 1, 2).double()
        for h in range(2):
            v, g = _grad(lambda x: 0.25 * O.pdice_loss(torch.softmax(x, 1), ref_pseudo[:, None].long()), logits[h])
            with torch.no_grad():
                s = torch.softmax(logits[h].double(), 1)
                sums = torch.cat([torch.tensor([v / 0.25], device=DEV, dtype=torch.float64),
                                  N * (s * t).sum((0, 2, 3)), N * t.sum((0, 2, 3)), N * (s * s).sum((0, 2, 3))])
            r["checks"][f"pd{h}"] = (_buf(step, f"pd{h}", (13,)), sums)
            r["loss"] += v
            r["g_reg"][h] = g
    return r


CASES = [  # (N, H, W, regime, labels)
    FULL + ("trained", "scribble"),
    FULL + ("init", "scribble"),
    FULL + ("saturated", "scribble"),
    (2, 32, 32, "trained", "dense"),           # fixture scale
    (9, 40, 100, "trained", "high"),           # H*W % 4 == 0, CRF tiles ragged both ways, one warp owns two samples in the finalizers
    (9, 40, 100, "init", "none"),
    (9, 40, 100, "saturated", "dense"),
]
HEAD_PARAMS = [(v,) + c for v in VARIANTS for c in CASES] + [("pce_tv", 1, 32, 32, "trained", "scribble")]


def _case_id(p):
    return f"{p[0]}-{p[1]}x{p[2]}x{p[3]}-{p[4]}-{p[5]}"


@pytest.mark.parametrize("variant,N,H,W,regime,labels", HEAD_PARAMS, ids=[_case_id(p) for p in HEAD_PARAMS])
def test_head_fp32_matches_fp64(variant, N, H, W, regime, labels):
    step = _step(variant, "fp32")
    heads = 2 if variant == "dmpls" else 1
    seed = 1000 * N + H + W
    logits = _logits(regime, N, H, W, seed, heads)
    image, label = _batch(labels, N, H, W, seed)
    loss, dl = step._head(logits, image, label, "t")
    torch.cuda.synchronize()
    ref = _reference(variant, step, logits, image, label, regime)

    # loss: NaN exactly when no pixel is labelled (torch's mean over nothing)
    if labels == "none":
        assert math.isnan(loss.item()) and math.isnan(ref["loss"])
        loss_err = 0.0
    else:
        loss_err = _rel(loss.item(), ref["loss"])
    buf_err = {name: _close(got, want) for name, (got, want) in ref["checks"].items()}
    unl = (label >= 4)[:, None].expand(N, 4, H, W)
    g_err, u_err = [], []
    for h in range(heads):
        d = dl[h]
        assert torch.isfinite(d).all()
        g_ref = ref["g_ce"][h] + (ref["g_reg"][h] if ref["g_reg"][h] is not None else 0.0)
        gmax = g_ref.abs().max().item()
        err = (d.double() - g_ref).abs().max().item()
        g_err.append(err / gmax if gmax > 0 else err)
        # the regulariser on its own: pCE adds exactly nothing on unlabelled pixels
        du = d[unl]
        if du.numel() == 0:                     # dense labels
            continue
        if ref["g_reg"][h] is None:
            assert (du == 0).all()
            continue
        gu = ref["g_reg"][h][unl]
        if gu.abs().max().item() < 1e-30:       # saturated softmax: the regulariser's logit gradient is below fp32's range
            assert du.abs().max().item() <= 1e-30
            continue
        u_err.append(rel_l2(du, gu))
    print(f"[head fp32 {_case_id((variant, N, H, W, regime, labels))}] loss err {loss_err:.2e}, "
          f"grad err {max(g_err):.2e} of max|g|, unlabelled regulariser rel-L2 {max(u_err, default=0.0):.2e}, "
          f"buffers {', '.join(f'{k} {v * 1e-5:.1e}' for k, v in buf_err.items())}")

    assert loss_err <= 1e-5
    if "w" in ref:
        assert _rel(step.cw_dev.item(), ref["w"]) < 1e-7
    for name, err in buf_err.items():           # in units of the 1e-5 tolerance
        assert err <= (10.0 if (name == "varstats" and regime == "init") else 1.0), (name, err)
    assert max(g_err) <= (1.2e-4 if (regime == "init" and labels == "none") else 1e-5)
    assert max(u_err, default=0.0) <= (4e-4 if (variant == "pce_variance" and regime == "init") else 1e-4)
    if "tv_gprobs" in ref:
        gp, gtv = ref["tv_gprobs"]
        unit = 1e-2 / max(1, gtv[1:].numel())
        nz = gtv.abs() > 0.5 * unit
        assert torch.equal(gp != 0, nz), "TV gradient support differs from torch's"
        assert (gtv[~nz].abs() < 1e-3 * unit).all()
        assert (gp[0] == 0).all(), "sample 0 is outside tv_loss(outputs_soft[1:])"
        if nz.any():
            assert ((gp[nz] - gtv[nz]).abs() / gtv[nz].abs()).max().item() <= 1e-6
    if "pseudo" in ref:
        assert torch.equal(*ref["pseudo"]), "pseudo labels differ from torch.argmax of the fp32 mix"


def test_variance_zero_std_gives_zero_gradient():
    """A sample whose image is 0 has v = img * p = 0: every standard deviation of the class-variance term is 0.  torch's std
    backward masks a zero result to a zero gradient instead of 0/0; the kernels do the same for that sample (losses.cu,
    variance_bwd_kernel) and keep the other samples' gradients."""
    N, H, W = 4, 32, 32
    step = _step("pce_variance", "fp32")
    logits = _logits("trained", N, H, W, 77, 1)
    image, label = _batch("scribble", N, H, W, 77)
    image[0] = 0.0
    step._head(logits, image, label, "t")
    torch.cuda.synchronize()
    gp = _buf(step, "gprobs0", (N, 4, H, W))
    st = _buf(step, "varstats", (N * 4 * 2 + N * 2,))
    assert (gp[0] == 0).all()
    assert (st[0:8] == 0).all() and (st[N * 8:N * 8 + 2] == 0).all()      # sample 0: class means / stds, mean / std over classes
    p = _buf(step, "probs0", (N, 4, H, W)).double().requires_grad_(True)
    (g,) = torch.autograd.grad(O.class_variance_loss(p, image.double()), p)
    assert (g[0] == 0).all()
    assert (gp[1:].double() - g[1:]).abs().max().item() <= 1e-5 * g[1:].abs().max().item()
    unl = (label[0] >= 4)[None].expand(4, H, W)
    assert (_buf(step, "dl0", (N, 4, H, W))[0][unl] == 0).all()


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_head_16bit_is_the_scaled_fp32_gradient(variant, precision):
    N, H, W = FULL
    heads = 2 if variant == "dmpls" else 1
    logits = _logits("trained", N, H, W, 4242, heads)
    image, label = _batch("scribble", N, H, W, 4242)
    s32, s16 = _step(variant, "fp32"), _step(variant, precision)
    l32, dl32 = s32._head(logits, image, label, "t")
    l16, dl16 = s16._head(logits, image, label, "t")
    torch.cuda.synchronize()
    assert l16.item() == l32.item()
    S = s16.ex.grad_scale_for(N, H, W)
    assert S == 2.0 ** round(math.log2(S)) and (S == 1.0) == (precision == "bf16")
    dt = torch.float16 if precision == "fp16" else torch.bfloat16
    for h in range(heads):
        kind, d16 = dl16[h]
        assert kind == "nhwc16" and d16.shape == (N, H, W, 16) and d16.dtype == dt
        assert (d16[..., 4:] == 0).all()
        want32 = (dl32[h] * S).permute(0, 2, 3, 1)
        want = want32.to(dt)
        got = d16[..., :4]
        assert torch.equal(got, want), (got != want).sum().item()
        if precision == "fp16":
            assert not torch.isinf(got).any()
            nz = want32 != 0
            flush = ((got == 0) & nz).sum().item() / max(1, nz.sum().item())
            print(f"[head fp16 {variant} dl{h}] S = 2^{int(math.log2(S))}, flushed {flush:.3e} of the nonzero elements")
            assert flush <= FP16_FLUSH_MAX[variant], flush


# ------------------------------------------------------------------------------------------------------------------------
# mean-teacher consistency (K13) and USTM's rot90
# ------------------------------------------------------------------------------------------------------------------------
UAMT_B, UAMT_T = 32, 8          # bench.py's UAMT batch: 64 images per GPU, half unlabelled


def _uamt_inputs(seed=5):
    B, T, H, W = UAMT_B, UAMT_T, 256, 256
    g = torch.Generator(device=DEV).manual_seed(seed)
    student = 2.0 * torch.randn(B, 4, H, W, generator=g, device=DEV)
    teacher = 2.0 * torch.randn(B, 4, H, W, generator=g, device=DEV)
    mc = 1.5 * torch.randn(T * B, 4, H, W, generator=g, device=DEV)      # every teacher pass distinct
    preds = F.softmax(mc.double(), dim=1).reshape(T, B, 4, H, W).mean(0)
    unc = -(preds * torch.log(preds + 1e-6)).sum(1)                       # train_uncertainty_aware_mean_teacher_2D.py:171-176
    return student, teacher, mc, unc


def _uamt(student, teacher, mc, thr, w):
    B, _, H, W = student.shape
    thr_dev = torch.tensor([thr], dtype=torch.float32, device=DEV)
    w_dev = torch.tensor([w], dtype=torch.float32, device=DEV)
    mask = torch.empty(B, H, W, dtype=torch.uint8, device=DEV)
    cst = torch.empty(3, device=DEV)
    dl = torch.empty_like(student)
    call("wsl_uamt_consistency_fwd", student, teacher, mc, UAMT_T, B, 4, H, W, thr_dev, 0.0, mask, cst, workspace("t_uamt"))
    call("wsl_uamt_consistency_bwd", student, teacher, mask, cst, w_dev, 0.0, B, 4, H, W, dl)
    torch.cuda.synchronize()
    return mask, cst, dl


def test_uamt_consistency_matches_fp64():
    student, teacher, mc, unc = _uamt_inputs()
    thr = torch.tensor(unc.median().item(), dtype=torch.float32).item()       # the median of the fp64 uncertainty, as fp32
    w = 0.37
    mask, cst, dl = _uamt(student, teacher, mc, thr, w)
    ref_mask = unc < thr
    far = (unc - thr).abs() > 1e-5
    assert torch.equal(mask.bool()[far], ref_mask[far])
    assert 0.3 < mask.float().mean().item() < 0.7
    m = mask.double()[:, None]
    s = student.double().requires_grad_(True)
    dist = O.softmax_mse(s, teacher.double())
    tot, cnt = (m * dist).sum(), mask.double().sum()
    loss = tot / (2 * cnt + 1e-16)
    (g,) = torch.autograd.grad(w * loss, s)
    for i, (a, b) in enumerate(((cst[0].item(), tot.item()), (cst[1].item(), cnt.item()), (cst[2].item(), loss.item()))):
        assert _rel(a, b) <= 1e-5, (i, a, b)
    e = rel_l2(dl, g)
    print(f"[uamt B={UAMT_B} T={UAMT_T}] mask on {mask.float().mean().item():.3f}, loss err {_rel(cst[2].item(), loss.item()):.2e}, "
          f"dlogits rel-L2 {e:.2e}")
    assert e <= 1e-5


def test_uamt_consistency_all_masked_off():
    student, teacher, mc, _ = _uamt_inputs(6)
    mask, cst, dl = _uamt(student, teacher, mc, -1.0, 0.5)
    assert (mask == 0).all()
    assert cst[0].item() == 0.0 and cst[1].item() == 0.0 and cst[2].item() == 0.0
    assert (dl == 0).all()


@pytest.mark.parametrize("S", [256, 37])
def test_rot90_bit_exact(S):
    g = torch.Generator(device=DEV).manual_seed(S)
    x = torch.randn(2, 4, S, S, generator=g, device=DEV)
    for k in range(4):
        want = torch.rot90(x, k, [2, 3])
        out = torch.empty_like(x)
        call("wsl_rot90", x, 8, S, k, 0, out)
        assert torch.equal(out, want), k
        acc0 = torch.randn(2, 4, S, S, generator=g, device=DEV)
        acc = acc0.clone()
        call("wsl_rot90", x, 8, S, k, 1, acc)
        assert torch.equal(acc, acc0 + want), k
        back = torch.empty_like(x)
        call("wsl_rot90", out, 8, S, (4 - k) % 4, 0, back)       # the rotate-back of USTMStep._body
        assert torch.equal(back, x), k


@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_ustm_gradient_is_pce_plus_rotated_back_consistency(k):
    """USTMStep._body: the logit gradient handed to backward() is the pCE gradient plus rot90(d consistency / d rot90(logits),
    -k), summed in place by the accumulating rot90."""
    B, hw = 2, 32
    torch.manual_seed(40 + k)
    student, teacher = UNet(1, 4).to(DEV).set_precision("fp32"), UNet(1, 4).to(DEV).set_precision("fp32")
    img, lab = O.synth_batch(B, hw, hw, seed=9, frac=0.1)
    img, lab = img.to(DEV), lab.to(DEV)
    step = USTMStep(student, teacher)
    step._ramps()
    step.ramp_dev[0] = 10.0                     # every pixel below the uncertainty threshold, weight 1: dr is not zero
    step.ramp_dev[1] = 1.0
    step._body(img, lab, None, k)
    torch.cuda.synchronize()
    Bf = lambda name, shape: step.ex.buf("ustm", name, shape, torch.float32)
    shp = (B, 4, hw, hw)
    d, dr, probs, st = Bf("dl", shp), Bf("dr", shp), Bf("probs", shp), Bf("stats", (2,))
    assert dr.abs().max().item() > 0
    pce = torch.empty(shp, device=DEV)
    call("wsl_head_bwd", probs, lab, st, None, 1.0, None, 0.0, B, 4, hw, hw, 4, pce, None, step.ex.dt)
    torch.cuda.synchronize()
    assert torch.equal(d, pce + torch.rot90(dr, -k, [2, 3]))


# ------------------------------------------------------------------------------------------------------------------------
# ticket reductions: run-to-run determinism and the ticket reset; the UNet_DS nearest resize
# ------------------------------------------------------------------------------------------------------------------------
def test_ticket_reductions_are_deterministic_at_full_size():
    """Every reduction launched twice back to back on the same workspace at 64x256x256: bit-identical results.  The outputs
    are poisoned with NaN in between, so a ticket left unreset (no block finalises on the second launch) shows."""
    N, H, W = FULL
    logits = _logits("trained", N, H, W, 99, 2)
    image, label = _batch("scribble", N, H, W, 99)
    probs = torch.softmax(logits[0], 1).contiguous()
    pseudo = torch.softmax(logits[1], 1).argmax(1).to(torch.uint8)
    student, teacher, mc, unc = _uamt_inputs(7)
    thr = torch.tensor([unc.median().item()], dtype=torch.float32, device=DEV)
    P = (N, 4, H, W)

    def run(name, outs, fn):
        res = []
        for _ in range(2):
            for o in outs:
                o.fill_(float("nan")) if o.is_floating_point() else o.fill_(7)
            fn()
            torch.cuda.synchronize()
            res.append([o.clone() for o in outs])
        for a, b in zip(*res):
            assert torch.equal(a, b) and (not a.is_floating_point() or not torch.isnan(a).any()), name

    o2, o1, o3, o13 = torch.empty(2, device=DEV), torch.empty(1, device=DEV), torch.empty(3, device=DEV), torch.empty(13, device=DEV)
    pr, gp = torch.empty(P, device=DEV), torch.empty(P, device=DEV)
    cent, vst = torch.empty(N * 4, device=DEV), torch.empty(N * 4 * 2 + N * 2, device=DEV)
    mask = torch.empty(32, H, W, dtype=torch.uint8, device=DEV)
    run("pce", [o2, pr], lambda: call("wsl_softmax_pce_fwd", logits[0], label, pr, N, 4, H, W, 4, o2, workspace("t_det")))
    run("crf", [o2, gp], lambda: call("wsl_gatedcrf_fwd", probs, image, gp, N, 4, H, W, 5, 6.0, 0.1, 1.0, o2, workspace("t_det")))
    run("ms", [o1, cent], lambda: call("wsl_mumford_shah_fwd", image, probs, N, 4, H, W, o1, cent, workspace("t_det")))
    run("pdice", [o13], lambda: call("wsl_pdice_fwd", probs, pseudo, None, float(N), N, 4, H, W, o13, workspace("t_det")))
    run("tv", [o1, gp], lambda: (gp.zero_(), call("wsl_tv_loss", probs, N * 4, H, W, 1e-2, gp, o1, workspace("t_det"))))
    run("entropy", [o1], lambda: call("wsl_entropy_fwd", probs, N, 4, H, W, o1, workspace("t_det")))
    run("variance", [o3, vst], lambda: call("wsl_class_variance_fwd", image, probs, N, 4, H, W, o3, vst, workspace("t_det")))
    run("uamt", [o3, mask], lambda: call("wsl_uamt_consistency_fwd", student, teacher, mc, UAMT_T, UAMT_B, 4, H, W, thr, 0.0,
                                          mask, o3, workspace("t_det")))


RESIZE = [(32, 32, 256, 256), (64, 64, 256, 256), (128, 128, 256, 256), (24, 24, 40, 40), (7, 7, 25, 25), (24, 7, 40, 25)]


@pytest.mark.parametrize("h,w,H,W", RESIZE, ids=[f"{a}x{b}-{c}x{d}" for a, b, c, d in RESIZE])
def test_nearest_resize_matches_interpolate(h, w, H, W):
    planes = 3 * 4
    g = torch.Generator(device=DEV).manual_seed(h * 1000 + W)
    x = torch.randn(1, planes, h, w, generator=g, device=DEV)
    out = torch.empty(1, planes, H, W, device=DEV)
    call("wsl_nearest_resize_fwd", x, planes, h, w, H, W, out)
    xr = x.clone().requires_grad_(True)
    y = F.interpolate(xr, size=(H, W))                        # mode='nearest', as Decoder_DS (networks/unet.py:177-185)
    assert torch.equal(out, y.detach())
    gy = torch.randint(-64, 64, (1, planes, H, W), generator=g, device=DEV).float() / 16     # dyadic: every sum is exact
    (gx,) = torch.autograd.grad(y, xr, gy)
    gsrc = torch.empty(1, planes, h, w, device=DEV)
    call("wsl_nearest_resize_bwd", gy, planes, h, w, H, W, gsrc)
    torch.cuda.synchronize()
    assert torch.equal(gsrc, gx)
