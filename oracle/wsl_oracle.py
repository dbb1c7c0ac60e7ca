"""CPU oracle for the WSL4MIS segmentation-training hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``wsl4mis_b200/`` may import this file; only
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of
``bench.py`` do, and there only as the checker / the timed CPU baseline.

This is a from-scratch *functional* restatement (plain torch fp32/fp64 ops on CPU tensors) of the
reference's per-step arithmetic.  The reference itself is pure PyTorch with no native code, so the
arithmetic lives in torch; the restatement is pinned against the unmodified reference modules by
``oracle/make_golden.py`` (runs in the build container where ``/root/reference`` exists) and the
fixtures it writes to ``tests/golden/`` (checked by ``tests/test_oracle_golden.py``).

Every function cites the reference ``file:line`` (relative to ``/root/reference/code``) it follows.
Parameter dictionaries use the reference's ``state_dict`` key names verbatim.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

FT = (16, 32, 64, 128, 256)            # networks/unet.py:291
ENC_DROP = (0.05, 0.1, 0.2, 0.3, 0.5)  # networks/unet.py:292
BN_EPS = 1e-5                          # nn.BatchNorm2d default, networks/unet.py:20
BN_MOM = 0.1
LRELU = 0.01                           # nn.LeakyReLU default, networks/unet.py:21


# ----------------------------------------------------------------------------------------------
# parameter construction
# ----------------------------------------------------------------------------------------------
def unet_param_shapes(in_chns: int, class_num: int, decoders: Sequence[str] = ("decoder",), ds: bool = False):
    """Ordered {state_dict key: shape} for UNet (decoders=('decoder',)) or UNet_CCT
    (decoders=('main_decoder','aux_decoder1')).  Order follows module registration order in
    networks/unet.py:71-121,286-298,327-339 so it equals ``reference_model.state_dict().keys()``."""
    shapes: Dict[str, Tuple[int, ...]] = {}

    def conv(prefix, cin, cout, k):
        shapes[f"{prefix}.weight"] = (cout, cin, k, k)
        shapes[f"{prefix}.bias"] = (cout,)

    def bn(prefix, c):
        shapes[f"{prefix}.weight"] = (c,)
        shapes[f"{prefix}.bias"] = (c,)
        shapes[f"{prefix}.running_mean"] = (c,)
        shapes[f"{prefix}.running_var"] = (c,)
        shapes[f"{prefix}.num_batches_tracked"] = ()

    def block(prefix, cin, cout):
        conv(f"{prefix}.0", cin, cout, 3)
        bn(f"{prefix}.1", cout)
        conv(f"{prefix}.4", cout, cout, 3)
        bn(f"{prefix}.5", cout)

    block("encoder.in_conv.conv_conv", in_chns, FT[0])
    for i in range(1, 5):
        block(f"encoder.down{i}.maxpool_conv.1.conv_conv", FT[i - 1], FT[i])
    for d in decoders:
        for j, (c1, c2) in enumerate(((FT[4], FT[3]), (FT[3], FT[2]), (FT[2], FT[1]), (FT[1], FT[0])), 1):
            conv(f"{d}.up{j}.conv1x1", c1, c2, 1)
            block(f"{d}.up{j}.conv.conv_conv", 2 * c2, c2)
        conv(f"{d}.out_conv", FT[0], class_num, 3)
        if ds:      # Decoder_DS registers the deep-supervision heads after out_conv (networks/unet.py:159-168); dp4 is never used
            for lvl in (4, 3, 2, 1):
                conv(f"{d}.out_conv_dp{lvl}", FT[lvl], class_num, 3)
    return shapes


def synth_params(in_chns: int, class_num: int, decoders: Sequence[str], seed: int,
                 dtype=torch.float32, ds: bool = False) -> Dict[str, torch.Tensor]:
    """Deterministic, torch-RNG-independent parameters (numpy RandomState stream, stable across
    versions) so golden fixtures only need to store a seed.  Scales mimic kaiming-uniform fan-in
    init; BN affine/running stats are randomised so every term of the BN formula is exercised."""
    import numpy as np

    rs = np.random.RandomState(seed)
    out: Dict[str, torch.Tensor] = {}
    for k, shp in unet_param_shapes(in_chns, class_num, decoders, ds).items():
        if k.endswith("num_batches_tracked"):
            out[k] = torch.zeros((), dtype=torch.long)
            continue
        if k.endswith("running_var"):
            a = rs.uniform(0.5, 1.5, size=shp)
        elif k.endswith("running_mean"):
            a = rs.uniform(-0.2, 0.2, size=shp)
        elif len(shp) == 4:
            fan_in = shp[1] * shp[2] * shp[3]
            b = math.sqrt(3.0 / fan_in) * 1.4
            a = rs.uniform(-b, b, size=shp)
        elif ".1." in k[-12:] or ".5." in k[-12:]:  # BN weight / bias
            a = rs.uniform(0.6, 1.4, size=shp) if k.endswith("weight") else rs.uniform(-0.3, 0.3, size=shp)
        else:  # conv bias
            a = rs.uniform(-0.1, 0.1, size=shp)
        out[k] = torch.from_numpy(np.ascontiguousarray(a)).to(dtype)
    return out


# ----------------------------------------------------------------------------------------------
# optional storage-precision emulation (used by the GPU parity tests to separate "kernel is wrong" from
# "bf16 storage costs precision"): QUANT rounds forward values AND the gradients flowing back through the
# same point to bf16 (or fp16, with the executor's loss scale), at exactly the tensors the executor stores in 16 bits (conv outputs Y, activations A,
# conv1x1 output T, upsample output U, channel-dropped features) and rounds the weights of the convolutions
# that run on the tensor cores.  QUANT = None (default) is the plain fp32 restatement of the reference.
# ----------------------------------------------------------------------------------------------
QUANT = None          # None | True / "bf16" | "fp16"
QUANT_SCALE = 1.0     # power-of-two loss scale the fp16 executor carries on every activation gradient (grad_scale_for)


def _qdtype():
    return torch.float16 if QUANT == "fp16" else torch.bfloat16


class _RoundBoth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(_qdtype()).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        if QUANT == "fp16":          # the stored value is fp16(g * scale); the scale is exact (power of two)
            return (g * QUANT_SCALE).to(torch.float16).to(g.dtype) / QUANT_SCALE
        return g.to(torch.bfloat16).to(g.dtype)


def _q(x):
    return x if QUANT is None else _RoundBoth.apply(x)


def _qw(w, x):
    """weights are 16-bit on the tcgen05 path: Cin % 16 == 0 and the map is a multiple of the 8x16 pixel tile"""
    if QUANT is None:
        return w
    tc = (w.shape[1] % 16 == 0) and (x.shape[-1] % 16 == 0) and (x.shape[-2] % 8 == 0)
    return w.to(_qdtype()).to(w.dtype) if tc else w


# ----------------------------------------------------------------------------------------------
# network forward (functional)
# ----------------------------------------------------------------------------------------------
def _apply_elem_dropout(x, p, training, mask):
    """nn.Dropout(p) (networks/unet.py:22).  ``mask`` (uint8/bool keep mask, same shape as x) makes
    it deterministic; otherwise torch's RNG is used like the reference does."""
    if not training or p == 0.0:
        return x
    if mask is None:
        return F.dropout(x, p, True)
    return x * mask.to(x.dtype) * (1.0 / (1.0 - p))


def conv_block(p, prefix, x, training, drop_p, masks=None, new_stats=None):
    """ConvBlock, networks/unet.py:13-29: conv3x3+bias -> BN -> LeakyReLU -> Dropout -> conv3x3 -> BN
    -> LeakyReLU.  Running statistics are not mutated in ``p``; updated values are written to
    ``new_stats`` (dict) when given."""
    for idx, bnidx, dp in ((0, 1, drop_p), (4, 5, 0.0)):
        x = _q(F.conv2d(x, _qw(p[f"{prefix}.{idx}.weight"], x), p[f"{prefix}.{idx}.bias"], padding=1))
        rm = p[f"{prefix}.{bnidx}.running_mean"].clone()
        rv = p[f"{prefix}.{bnidx}.running_var"].clone()
        x = F.batch_norm(x, rm, rv, p[f"{prefix}.{bnidx}.weight"], p[f"{prefix}.{bnidx}.bias"],
                         training, BN_MOM, BN_EPS)
        if new_stats is not None and training:
            new_stats[f"{prefix}.{bnidx}.running_mean"] = rm
            new_stats[f"{prefix}.{bnidx}.running_var"] = rv
        x = F.leaky_relu(x, LRELU)
        if dp > 0.0:
            x = _apply_elem_dropout(x, dp, training, None if masks is None else masks.get(f"{prefix}.3"))
        x = _q(x)
    return x


def encoder_forward(p, x, training, masks=None, new_stats=None):
    """Encoder.forward, networks/unet.py:92-98 (+ DownBlock :32-44: MaxPool2d(2) then ConvBlock)."""
    feats = [conv_block(p, "encoder.in_conv.conv_conv", x, training, ENC_DROP[0], masks, new_stats)]
    for i in range(1, 5):
        x_in = F.max_pool2d(feats[-1], 2)
        feats.append(conv_block(p, f"encoder.down{i}.maxpool_conv.1.conv_conv", x_in, training,
                                ENC_DROP[i], masks, new_stats))
    return feats


def decoder_forward(p, dname, feats, training, new_stats=None):
    """Decoder.forward, networks/unet.py:123-135; UpBlock (bilinear branch) :63-68:
    conv1x1 -> bilinear x2 (align_corners=True) -> cat([skip, up]) -> ConvBlock(p=0)."""
    x = feats[4]
    for j, skip in enumerate((feats[3], feats[2], feats[1], feats[0]), 1):
        t = _q(F.conv2d(x, _qw(p[f"{dname}.up{j}.conv1x1.weight"], x), p[f"{dname}.up{j}.conv1x1.bias"]))
        t = _q(F.interpolate(t, scale_factor=2, mode="bilinear", align_corners=True))
        x = conv_block(p, f"{dname}.up{j}.conv.conv_conv", torch.cat([skip, t], 1), training, 0.0,
                       None, new_stats)
    return F.conv2d(x, _qw(p[f"{dname}.out_conv.weight"], x), p[f"{dname}.out_conv.bias"], padding=1)


def unet_forward(p, x, training=True, masks=None, new_stats=None):
    """UNet.forward, networks/unet.py:300-303."""
    return decoder_forward(p, "decoder", encoder_forward(p, x, training, masks, new_stats), training, new_stats)


def channel_dropout(x, keep):
    """Dropout(x, p=0.5) = F.dropout2d with training=True always (networks/unet.py:254-256, F5):
    per-(n,c) Bernoulli keep mask, survivors scaled by 2.  ``keep`` is a [N,C] 0/1 tensor."""
    if keep is None:
        return F.dropout2d(x, 0.5)
    return _q(x * (keep.to(x.dtype) * 2.0)[:, :, None, None])


def unet_cct_forward(p, x, training=True, masks=None, chan_keep=None, new_stats=None):
    """UNet_CCT.forward, networks/unet.py:341-346.  ``chan_keep`` is a list of five [N,C_i] keep masks
    for the aux branch (None -> torch RNG, as the reference)."""
    feats = encoder_forward(p, x, training, masks, new_stats)
    main = decoder_forward(p, "main_decoder", feats, training, new_stats)
    aux_feats = [channel_dropout(f, None if chan_keep is None else chan_keep[i]) for i, f in enumerate(feats)]
    aux = decoder_forward(p, "aux_decoder1", aux_feats, training, new_stats)
    return main, aux


# ----------------------------------------------------------------------------------------------
# other heads of the family (SURVEY 8(f) rank 4; restated ahead of the product, which does not build them yet)
# ----------------------------------------------------------------------------------------------
def decoder_ds_forward(p, dname, feats, shape, training, new_stats=None):
    """Decoder_DS.forward, networks/unet.py:169-190: the Decoder plus a 3x3 class head on the output of up1/up2/up3, each
    resized to the input size with F.interpolate's default nearest mode.  Returns (dp0, dp1, dp2, dp3)."""
    x = feats[4]
    heads = {}
    for j, skip in enumerate((feats[3], feats[2], feats[1], feats[0]), 1):
        t = _q(F.conv2d(x, _qw(p[f"{dname}.up{j}.conv1x1.weight"], x), p[f"{dname}.up{j}.conv1x1.bias"]))
        t = _q(F.interpolate(t, scale_factor=2, mode="bilinear", align_corners=True))
        x = conv_block(p, f"{dname}.up{j}.conv.conv_conv", torch.cat([skip, t], 1), training, 0.0, None, new_stats)
        if j < 4:
            lvl = 4 - j                                                                   # up1 -> dp3, up2 -> dp2, up3 -> dp1
            dp = F.conv2d(x, _qw(p[f"{dname}.out_conv_dp{lvl}.weight"], x), p[f"{dname}.out_conv_dp{lvl}.bias"], padding=1)
            heads[lvl] = F.interpolate(dp, shape)
    dp0 = F.conv2d(x, _qw(p[f"{dname}.out_conv.weight"], x), p[f"{dname}.out_conv.bias"], padding=1)
    return dp0, heads[1], heads[2], heads[3]


def unet_ds_forward(p, x, training=True, masks=None, new_stats=None):
    """UNet_DS.forward, networks/unet.py:319-324."""
    feats = encoder_forward(p, x, training, masks, new_stats)
    return decoder_ds_forward(p, "decoder", feats, x.shape[2:], training, new_stats)


def feature_noise(x, noise):
    """FeatureNoise.forward, networks/unet.py:270-283: one uniform(-0.3, 0.3) tensor of shape x.shape[1:] shared by the batch,
    x * noise + x.  ``noise`` is that tensor (the reference draws it from torch's global RNG)."""
    return _q(x * noise.unsqueeze(0) + x)


def unet_cct_3h_forward(p, x, training=True, masks=None, chan_keep=None, noises=None, new_stats=None):
    """UNet_CCT_3H.forward, networks/unet.py:363-371, AS WRITTEN: the third head runs ``aux_decoder1`` again on the
    noise-perturbed features (:370) -- ``aux_decoder2`` owns parameters but never runs."""
    feats = encoder_forward(p, x, training, masks, new_stats)
    main = decoder_forward(p, "main_decoder", feats, training, new_stats)
    aux1 = decoder_forward(p, "aux_decoder1", [channel_dropout(f, None if chan_keep is None else chan_keep[i])
                                               for i, f in enumerate(feats)], training, new_stats)
    aux2 = decoder_forward(p, "aux_decoder1", [feature_noise(f, noises[i]) for i, f in enumerate(feats)], training, new_stats)
    return main, aux1, aux2


# ----------------------------------------------------------------------------------------------
# PNet2D (networks/pnet.py:87-122; net_factory builds PNet2D(in_chns, class_num, 64, [1, 2, 4, 8, 16]))
# ----------------------------------------------------------------------------------------------
PNET_RATIOS = (1, 2, 4, 8, 16)


def pnet_param_shapes(in_chns: int, out_chns: int, nf: int = 64):
    """Ordered {state_dict key: shape} of PNet2D: per PNetBlock conv1, conv2, in1, in2 (pnet.py:25-32), then catblock.conv1/2
    (:49-52), out.conv1/2 (:68-71)."""
    shapes: Dict[str, Tuple[int, ...]] = {}

    def conv(prefix, cin, cout, k):
        shapes[f"{prefix}.weight"] = (cout, cin, k, k)
        shapes[f"{prefix}.bias"] = (cout,)

    def bn(prefix, c):
        for nm, shp in (("weight", (c,)), ("bias", (c,)), ("running_mean", (c,)), ("running_var", (c,)), ("num_batches_tracked", ())):
            shapes[f"{prefix}.{nm}"] = shp

    for b in range(1, 6):
        conv(f"block{b}.conv1", in_chns if b == 1 else nf, nf, 3)
        conv(f"block{b}.conv2", nf, nf, 3)
        bn(f"block{b}.in1", nf)
        bn(f"block{b}.in2", nf)
    conv("catblock.conv1", 5 * nf, 5 * nf, 1)
    conv("catblock.conv2", 5 * nf, 2 * nf, 1)
    conv("out.conv1", 2 * nf, nf, 1)
    conv("out.conv2", nf, out_chns, 1)
    return shapes


def pnet_synth_params(in_chns: int, out_chns: int, seed: int, nf: int = 64) -> Dict[str, torch.Tensor]:
    """numpy-stream parameters for PNet2D (same recipe as synth_params)."""
    import numpy as np
    rs = np.random.RandomState(seed)
    out: Dict[str, torch.Tensor] = {}
    for k, shp in pnet_param_shapes(in_chns, out_chns, nf).items():
        if k.endswith("num_batches_tracked"):
            out[k] = torch.zeros((), dtype=torch.long)
            continue
        if k.endswith("running_var"):
            a = rs.uniform(0.5, 1.5, size=shp)
        elif k.endswith("running_mean"):
            a = rs.uniform(-0.2, 0.2, size=shp)
        elif len(shp) == 4:
            b = math.sqrt(3.0 / (shp[1] * shp[2] * shp[3])) * 1.4
            a = rs.uniform(-b, b, size=shp)
        elif ".in1." in k or ".in2." in k:
            a = rs.uniform(0.6, 1.4, size=shp) if k.endswith("weight") else rs.uniform(-0.3, 0.3, size=shp)
        else:
            a = rs.uniform(-0.1, 0.1, size=shp)
        out[k] = torch.from_numpy(np.ascontiguousarray(a)).float()
    return out


def pnet2d_forward(p, x, training=True, chan_keep=None, new_stats=None):
    """PNet2D.forward (pnet.py:112-122): five PNetBlocks (:34-41: dilated conv3x3 -> BN -> LeakyReLU, twice; dilation = padding =
    ratio), concat of the five block outputs, ConcatBlock (:54-59: conv1x1 -> LeakyReLU -> conv1x1 -> LeakyReLU), OutPutBlock
    (:75-81: Dropout2d(0.3) -> conv1x1 -> LeakyReLU -> Dropout2d(0.3) -> conv1x1).  chan_keep: the two [N, C] keep masks of the
    Dropout2d layers (None -> torch RNG, like the reference)."""
    feats = []
    for b, r in enumerate(PNET_RATIOS, 1):
        for cv, bnn in (("conv1", "in1"), ("conv2", "in2")):
            x = _q(F.conv2d(x, _qw(p[f"block{b}.{cv}.weight"], x), p[f"block{b}.{cv}.bias"], padding=r, dilation=r))
            rm, rv = p[f"block{b}.{bnn}.running_mean"].clone(), p[f"block{b}.{bnn}.running_var"].clone()
            x = F.batch_norm(x, rm, rv, p[f"block{b}.{bnn}.weight"], p[f"block{b}.{bnn}.bias"], training, BN_MOM, BN_EPS)
            if new_stats is not None and training:
                new_stats[f"block{b}.{bnn}.running_mean"], new_stats[f"block{b}.{bnn}.running_var"] = rm, rv
            x = _q(F.leaky_relu(x, LRELU))
        feats.append(x)
    x = torch.cat(feats, 1)
    x = _q(F.leaky_relu(_q(F.conv2d(x, _qw(p["catblock.conv1.weight"], x), p["catblock.conv1.bias"])), LRELU))
    x = _q(F.leaky_relu(_q(F.conv2d(x, _qw(p["catblock.conv2.weight"], x), p["catblock.conv2.bias"])), LRELU))

    def drop2d(t, keep):
        if not training:
            return t
        if keep is None:
            return F.dropout2d(t, 0.3, True)
        return _q(t * (keep.to(t.dtype) * (1.0 / 0.7))[:, :, None, None])

    x = drop2d(x, None if chan_keep is None else chan_keep[0])
    x = _q(F.leaky_relu(_q(F.conv2d(x, _qw(p["out.conv1.weight"], x), p["out.conv1.bias"])), LRELU))
    x = drop2d(x, None if chan_keep is None else chan_keep[1])
    return F.conv2d(x, _qw(p["out.conv2.weight"], x), p["out.conv2.bias"])


# ----------------------------------------------------------------------------------------------
# losses
# ----------------------------------------------------------------------------------------------
def pce_loss(logits, label, ignore_index=4):
    """CrossEntropyLoss(ignore_index=4)(outputs, label.long()), constructed at
    train_weakly_supervised_pCE_2D.py:81 and called at :100.  Mean over labelled pixels; NaN when
    no pixel is labelled (torch semantics)."""
    return F.cross_entropy(logits, label.long(), ignore_index=ignore_index)


def gated_crf_loss(y, image, radius=5, sigma_xy=6.0, sigma_rgb=0.1, weight=1.0):
    """ModelLossSemsegGatedCRF.forward for the argument pattern every WSL4MIS script uses
    (utils/gate_crf_loss.py:20-117 with kernels_desc=[{'weight':1,'xy':6,'rgb':0.1}], radius 5, no
    masks, Potts compatibility; called at train_weakly_supervised_pCE_GatedCRFLoss_2D.py:115-122).

    Restated without F.unfold: loop over the (2r+1)^2-1 offsets on zero-padded tensors.  Zero padding
    of the *features* (gate_crf_loss.py:188) means an out-of-bounds neighbour has xy=(0,0)/sigma and
    intensity 0, so its kernel value is non-zero and is counted in ``kernels.sum()`` (:99) while
    contributing nothing to the pairwise product (SURVEY F10)."""
    N, C, H, W = y.shape
    dt = y.dtype
    xs = torch.arange(W, dtype=dt, device=y.device).view(1, 1, 1, W).expand(N, 1, H, W) / sigma_xy      # :174-181, :154
    ys = torch.arange(H, dtype=dt, device=y.device).view(1, 1, H, 1).expand(N, 1, H, W) / sigma_xy
    inten = F.adaptive_avg_pool2d(image.to(dt), (H, W)) / sigma_rgb                      # :127-132
    feat = torch.cat([xs, ys, inten], 1)
    r = radius
    fpad = F.pad(feat, (r, r, r, r))
    ypad = F.pad(y, (r, r, r, r))
    ksum = torch.zeros((), dtype=dt)
    pair = torch.zeros((), dtype=dt)
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dy == 0 and dx == 0:
                continue                                                                # centre := 0, :171
            fn = fpad[:, :, r + dy:r + dy + H, r + dx:r + dx + W]
            k = weight * torch.exp(-0.5 * ((fn - feat) ** 2).sum(1, keepdim=True))       # :168-170
            yn = ypad[:, :, r + dy:r + dy + H, r + dx:r + dx + W]
            ksum = ksum + k.sum()
            pair = pair + (k * yn * y).sum()
    return (ksum - pair) / (N * H * W)                                                  # :63, :97-99, :116


def gated_crf_loss_unfold(y, image, radius=5, sigma_xy=6.0, sigma_rgb=0.1, weight=1.0):
    """Same quantity as ``gated_crf_loss`` computed the way the reference does it (utils/gate_crf_loss.py:59-99,
    134-188): im2col (F.unfold, zero padded) of the scaled features and of the predictions, Gaussian of the
    feature differences with the centre tap zeroed, Potts shortcut.  This is the formulation timed as the CPU
    baseline (it is the reference's own algorithm and memory behaviour: the (2r+1)^2-fold unfold is materialised)."""
    N, C, H, W = y.shape
    d = 2 * radius + 1
    dt = y.dtype
    xs = torch.arange(W, dtype=dt, device=y.device).view(1, 1, 1, W).expand(N, 1, H, W) / sigma_xy
    ys = torch.arange(H, dtype=dt, device=y.device).view(1, 1, H, 1).expand(N, 1, H, W) / sigma_xy
    feat = torch.cat([xs, ys, F.adaptive_avg_pool2d(image.to(dt), (H, W)) / sigma_rgb], 1)
    fu = F.unfold(feat, d, 1, radius).view(N, 3, d, d, H, W)
    diff = fu - fu[:, :, radius, radius].view(N, 3, 1, 1, H, W)
    k = weight * torch.exp((-0.5 * diff * diff).sum(1, keepdim=True))
    k[:, :, radius, radius] = 0
    yu = F.unfold(y, d, 1, radius).view(N, C, d, d, H, W)
    prod = (k * yu).view(N, C, d * d, H, W).sum(2)
    return (k.sum() - (prod * y).sum()) / (N * H * W)


def mumford_shah_loss(image, prob):
    """MumfordShah_Loss.forward(image, prediction), utils/losses.py:275-309, as written: the image is
    passed as ``output`` and the softmax as ``target`` (SURVEY F11)."""
    loss = prob.new_zeros(())
    isum = image.sum((2, 3))                                      # :286-287 denominator
    for k in range(prob.shape[1]):
        t = prob[:, k:k + 1].expand(-1, image.shape[1], -1, -1)
        cent = (t * image).sum((2, 3)) / isum
        lvl = t - cent[:, :, None, None]
        loss = loss + (lvl * lvl * image).sum()
    dh = (prob[:, :, 1:, :] - prob[:, :, :-1, :]).abs().sum()    # gradientLoss2d :296-304 ('l1')
    dw = (prob[:, :, :, 1:] - prob[:, :, :, :-1]).abs().sum()
    return loss + dh + dw


def pdice_loss(prob, target, n_classes=4, ignore_index=4):
    """pDLoss.forward, utils/losses.py:195-232.  ``target`` is [N,1,H,W] integer.

    As written in the reference the ignore mask keeps its channel dim ([N,1,H,W], :219-220) while the
    per-class score/target slices are [N,H,W] (:229), so ``score * target * ignore_mask`` (:209-211)
    broadcasts to [N,N,H,W]: every per-pixel product is multiplied by the *batch-summed* mask at that
    pixel location, M[h,w] = sum_a mask[a,h,w] (= N when nothing is ignored, as in the DMPLS script
    where the target is an argmax map).  Reproduced as written (found by the golden fixtures)."""
    keep = (target != ignore_index).to(prob.dtype)[:, 0]           # [N,H,W]
    msum = keep.sum(0, keepdim=True)                                # [1,H,W]  batch-summed mask
    loss = prob.new_zeros(())
    for i in range(n_classes):
        t = (target == i).to(prob.dtype)[:, 0]
        s = prob[:, i]
        inter = (s * t * msum).sum()
        ysum = (t * t * msum).sum()
        zsum = (s * s * msum).sum()
        loss = loss + (1 - (2 * inter + 1e-5) / (zsum + ysum + 1e-5))
    return loss / n_classes


def dice_loss(prob, target, n_classes=4):
    """DiceLoss.forward (softmax=False, weight=None), utils/losses.py:156-192 (no mask, plain sums)."""
    loss = prob.new_zeros(())
    for i in range(n_classes):
        t = (target == i).to(prob.dtype)[:, 0]
        s = prob[:, i]
        loss = loss + (1 - (2 * (s * t).sum() + 1e-5) / ((s * s).sum() + (t * t).sum() + 1e-5))
    return loss / n_classes


def mix_pseudo_label(p1, p2, beta):
    """argmax(beta*p1 + (1-beta)*p2, dim=1), train_weakly_supervised_segmentation_pCE_ours_proposed.py:119-120."""
    return torch.argmax(beta * p1.detach() + (1.0 - beta) * p2.detach(), dim=1)


def tv_loss(prob):
    """tv_loss, train_weakly_supervised_pCE_TV_2D.py:58-65."""
    mn = -F.max_pool2d(-prob, (3, 3), 1, 1)
    contour = torch.relu(F.max_pool2d(mn, (3, 3), 1, 1) - mn)
    return contour.abs().mean()


def entropy_minimization(prob):
    """entropy_minmization, utils/losses.py:235-239."""
    return (-(prob * torch.log(prob + 1e-6)).sum(1)).mean()


def entropy_loss(prob, C=4):
    """losses.entropy_loss, utils/losses.py:30-36 (as called at train_weakly_supervised_pCE_Entropy_Mini_2D.py:99)."""
    return (-(prob * torch.log(prob + 1e-6)).sum(1) / math.log(C)).mean()


def class_variance_loss(prob, img):
    """inter_class_variance(prob, img) - intra_class_variance(prob, img),
    train_weakly_supervised_pCE_Inter&Intra_Class_2D.py:30-36,114."""
    v = img * prob
    intra = torch.std(v, dim=[2, 3]).mean()
    inter = torch.std(torch.mean(v, dim=[2, 3]), dim=1).mean()
    return inter - intra


def softmax_mse(a_logits, b_logits):
    """softmax_mse_loss (sigmoid=False), utils/losses.py:65-82."""
    return (F.softmax(a_logits, 1) - F.softmax(b_logits, 1)) ** 2


# ----------------------------------------------------------------------------------------------
# step bodies (loss composition) and the optimiser
# ----------------------------------------------------------------------------------------------
CRF_IMPL = "loop"   # "unfold" = the reference's materialising formulation (used for CPU timing)


def step_loss_pce_gatedcrf(logits, image, label):
    """train_weakly_supervised_pCE_GatedCRFLoss_2D.py:111-123."""
    soft = torch.softmax(logits, 1)
    ce = pce_loss(logits, label)
    crf = gated_crf_loss_unfold(soft, image) if CRF_IMPL == "unfold" else gated_crf_loss(soft, image)
    return ce + 0.1 * crf, ce, crf


def step_loss_dmpls(logits1, logits2, label, beta):
    """train_weakly_supervised_segmentation_pCE_ours_proposed.py:108-125."""
    s1, s2 = torch.softmax(logits1, 1), torch.softmax(logits2, 1)
    ce = 0.5 * (pce_loss(logits1, label) + pce_loss(logits2, label))
    pseudo = mix_pseudo_label(s1, s2, beta).unsqueeze(1)
    pse = 0.5 * (pdice_loss(s1, pseudo) + pdice_loss(s2, pseudo))
    return ce + 0.5 * pse, ce, pse, pseudo[:, 0]


def step_loss_pce_ms(logits, image, label):
    """train_weakly_supervised_pCE_MumfordShah_Loss_2D.py:98-103."""
    soft = torch.softmax(logits, 1)
    ce = pce_loss(logits, label)
    ms = mumford_shah_loss(image, soft)
    return ce + 1e-6 * ms, ce, ms


def step_loss_pce_tv(logits, label):
    """train_weakly_supervised_pCE_TV_2D.py:109-114 (tv on outputs_soft[1:], batch slice, F12)."""
    soft = torch.softmax(logits, 1)
    ce = pce_loss(logits, label)
    tv = tv_loss(soft[1:])
    return ce + 1e-2 * tv, ce, tv


def sigmoid_rampup(current, rampup_length):
    """utils/ramps.py:19-26."""
    if rampup_length == 0:
        return 1.0
    cur = min(max(float(current), 0.0), float(rampup_length))
    ph = 1.0 - cur / rampup_length
    return float(math.exp(-5.0 * ph * ph))


def uamt_losses(out_l, out_u, ema_out, mc_logits, label_l, iter_num, max_iterations, consistency=0.1,
                consistency_rampup=200.0, T=8):
    """Loss composition of train_uncertainty_aware_mean_teacher_2D.py:151-190.
    out_l / out_u: student logits on the labelled / unlabelled half; ema_out: teacher logits on the noisy unlabelled
    inputs (:157-158); mc_logits: the [T*B,4,H,W] buffer of the T/2 teacher calls on the twice-repeated batch (:164-170).
    label_l is dense (uint8/int64, no ignore_index: ce_loss = CrossEntropyLoss() at :127)."""
    B = out_u.shape[0]
    preds = F.softmax(mc_logits, dim=1).reshape(T, B, *mc_logits.shape[1:]).mean(0)            # :171-173
    uncertainty = -(preds * torch.log(preds + 1e-6)).sum(1, keepdim=True)                     # :175-176
    soft_l = torch.softmax(out_l, 1)
    loss_ce = F.cross_entropy(out_l, label_l.long())                                          # :178
    loss_dice = dice_loss(soft_l, label_l.long().unsqueeze(1))                                # :179
    supervised = 0.5 * (loss_dice + loss_ce)                                                  # :180
    cw = consistency * sigmoid_rampup(iter_num // 300, consistency_rampup)                    # :73-75, :181-182
    dist = softmax_mse(out_u, ema_out)                                                        # :183-184
    threshold = (0.75 + 0.25 * sigmoid_rampup(iter_num, max_iterations)) * math.log(2)        # :185-186
    mask = (uncertainty < threshold).float()                                                  # :187
    cons = (mask * dist).sum() / (2 * mask.sum() + 1e-16)                                     # :188-189
    return supervised + cw * cons, supervised, cons, mask, cw, threshold                      # :191


def ustm_losses(out, ema_out, mc_logits, label, rot_times, iter_num, max_iterations, T=8):
    """Loss composition of train_weakly_supervised_ustm_2D.py:119-157: pCE on the scribbles + uncertainty-masked consistency
    between rot90(student logits) and the teacher's logits on the rotated noisy input."""
    B = out.shape[0]
    preds = F.softmax(mc_logits, dim=1).reshape(T, B, *mc_logits.shape[1:]).mean(0)
    uncertainty = -(preds * torch.log(preds + 1e-6)).sum(1, keepdim=True)
    ce = pce_loss(out, label)                                                                  # :120-121
    cw = 1.0 * sigmoid_rampup(iter_num // 1000, 60)                                            # :55-57,147-148
    dist = softmax_mse(torch.rot90(out, rot_times, [2, 3]), ema_out)                           # :150-152
    threshold = (0.75 + 0.25 * sigmoid_rampup(iter_num, max_iterations)) * math.log(2)         # :153-154
    mask = (uncertainty < threshold).float()
    cons = (mask * dist).sum() / (2 * mask.sum() + 1e-16)                                      # :155-157
    return ce + cw * cons, ce, cons, mask, cw, threshold


def ema_update(ema_params, params, alpha, global_step):
    """update_ema_variables, train_weakly_supervised_ustm_2D.py:61-65 (parameters only, buffers untouched)."""
    a = min(1 - 1 / (global_step + 1), alpha)
    for k in ema_params:
        if ema_params[k].is_floating_point() and "running" not in k:
            ema_params[k] = ema_params[k] * a + (1 - a) * params[k]
    return a


def sgd_step(params, grads, moms, lr, momentum=0.9, weight_decay=1e-4):
    """optim.SGD(lr, momentum=0.9, weight_decay=1e-4).step(), train_weakly_supervised_pCE_2D.py:79-80,104.
    torch semantics: g += wd*w; first step buf = g, afterwards buf = mu*buf + g; w -= lr*buf.
    ``moms[k] is None`` marks the first step."""
    for k in params:
        g = grads[k] + weight_decay * params[k]
        moms[k] = g.clone() if moms.get(k) is None else moms[k] * momentum + g
        params[k] = params[k] - lr * moms[k]


def poly_lr(base_lr, iter_num, max_iterations):
    """train_weakly_supervised_pCE_2D.py:106-108 (applied after the step, using the pre-increment iter)."""
    return base_lr * (1.0 - iter_num / max_iterations) ** 0.9


# ----------------------------------------------------------------------------------------------
# synthetic batch (SURVEY 8(d))
# ----------------------------------------------------------------------------------------------
def synth_batch(n, h=256, w=256, seed=2022, frac=0.03, dense=False):
    g = torch.Generator().manual_seed(seed)
    image = torch.rand(n, 1, h, w, generator=g)
    if dense:
        label = torch.randint(0, 4, (n, h, w), generator=g, dtype=torch.uint8)
    else:
        label = torch.full((n, h, w), 4, dtype=torch.uint8)
        m = torch.rand(n, h, w, generator=g) < frac
        vals = torch.randint(0, 4, (int(m.sum()),), generator=g, dtype=torch.uint8)
        label[m] = vals
        label[0, 0, 0] = 1  # at least one labelled pixel
    return image, label


def full_step(p, image, label, variant="pce_gatedcrf", cct=False, masks=None, chan_keep=None, beta=0.5):
    """One forward+loss+backward of a BASELINE config on CPU.  Returns (loss, grads dict, outputs)."""
    leaves = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in p.items()}
    if cct:
        main, aux = unet_cct_forward(leaves, image, True, masks, chan_keep)
    else:
        main, aux = unet_forward(leaves, image, True, masks), None
    if variant == "pce":
        loss = pce_loss(main, label)
    elif variant == "pce_gatedcrf":
        loss = step_loss_pce_gatedcrf(main, image, label)[0]
    elif variant == "pce_ms":
        loss = step_loss_pce_ms(main, image, label)[0]
    elif variant == "pce_tv":
        loss = step_loss_pce_tv(main, label)[0]
    elif variant == "dmpls":
        loss = step_loss_dmpls(main, aux, label, beta)[0]
    elif variant == "pce_entropy":       # train_weakly_supervised_pCE_Entropy_Mini_2D.py:97-102
        loss = pce_loss(main, label) + 0.1 * entropy_loss(torch.softmax(main, 1), 4)
    elif variant.startswith("pce_variance"):   # ...Inter&Intra_Class_2D.py:112-118, weight passed as "pce_variance:<w>"
        w = float(variant.split(":")[1]) if ":" in variant else 0.1
        loss = pce_loss(main, label) + w * class_variance_loss(torch.softmax(main, 1), image)
    else:
        raise ValueError(variant)
    names = [k for k, v in leaves.items() if v.requires_grad]
    gs = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    grads = {k: (g if g is not None else torch.zeros_like(leaves[k])) for k, g in zip(names, gs)}
    return loss.detach(), grads, (main.detach(), None if aux is None else aux.detach())
