"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by the product package `dinounet_b200`).

A functional, pure-PyTorch CPU restatement of the reference's Dino U-Net *forward* path,
written against a flat state dict that uses the reference's own parameter names.  It is
the checker for the hand-written sm_100a kernels; only `tests/`, `__graft_entry__.smoke()`
and `bench.py`'s cpu_baseline / `--impl reference` legs may import it.

Parity pin: on one host the restatement is bit-identical (fp32, CPU) to the REAL reference
forward imported through `oracle/ref_loader.py`; `tests/test_oracle_vs_reference.py` and
`tests/test_oracle_golden.py` hold it to the reference's outputs stored in `tests/golden/*.npz`
(made by `oracle/make_golden.py` and `oracle/make_golden_reference_pins.py`) within fp32
reduction-order noise.

Reference locations followed (all relative to /root/reference):
  DinoUNet.forward                      dinounet_training.py:786-804
  DINOv3EncoderAdapter.forward          dinounet_training.py:489-511
  FAPM / SE / DWSep / LearnableUpsample dinounet_training.py:419-441, 222-225, 241-246, 255-264
  UNetDecoder.forward                   dinounet_training.py:603-629
  DINOv3_Adapter.forward & friends      dinounet/dinov3/eval/segmentation/models/backbone/dinov3_adapter.py:40-484
  MSDeformAttn / core sampling          dinounet/dinov3/eval/segmentation/models/utils/ms_deform_attn.py:71-216
  DinoVisionTransformer taps            dinounet/dinov3/models/vision_transformer.py:186-216,265-318
  attention / rope / block / ffn / ls   dinounet/dinov3/layers/{attention.py:16-118, block.py:190-196,
                                        ffn_layers.py:43-77, layer_scale.py:28-29, patch_embed.py:64-76,
                                        rope_position_encoding.py:57-121}
  variant hyper-parameters              dinounet/dinov3/hub/backbones.py:201-237,279-315,318-371,452-494
  third-party conv blocks               dynamic-network-architectures 0.4.x StackedConvBlocks (not vendored)
"""
from __future__ import annotations

import math
import zlib
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# ----------------------------------------------------------------------------- configs
@dataclass(frozen=True)
class VariantCfg:
    name: str
    dim: int
    depth: int
    heads: int
    ffn: str            # "mlp" | "swiglu"
    ffn_hidden: int
    qkv_bias: bool
    taps: Tuple[int, ...]
    local_cls_norm: bool = False


VARIANTS: Dict[str, VariantCfg] = {
    # hub/backbones.py:201-237 ; interaction indexes dinounet_training.py:36-41
    "dinounet_s": VariantCfg("dinounet_s", 384, 12, 6, "mlp", 1536, True, (2, 5, 8, 11)),
    "dinounet_b": VariantCfg("dinounet_b", 768, 12, 12, "mlp", 3072, True, (2, 5, 8, 11)),
    "dinounet_l": VariantCfg("dinounet_l", 1024, 24, 16, "mlp", 4096, True, (4, 11, 17, 23)),
    # swiglu64, ffn_ratio 3 -> int(4096*3*2/3) aligned to 64 = 8192 (ffn_layers.py:67-68)
    "dinounet_7b": VariantCfg("dinounet_7b", 4096, 40, 32, "swiglu", 8192, False, (9, 19, 29, 39), True),
    # TEST-ONLY miniature of the 7B recipe (SwiGLU-64 with ffn_ratio 3, head_dim 128, no qkv bias, untied local cls norm):
    # exercises exactly the code paths that differ from s/b/l at a size the CPU oracle and the goldens can afford.
    "dinounet_7b_tiny": VariantCfg("dinounet_7b_tiny", 1024, 4, 8, "swiglu", 2048, False, (0, 1, 2, 3), True),
}

FEATURES = (32, 64, 128, 256)      # plans features_per_stage (SURVEY.md §8 A0)
RANK = 256                          # FAPM rank (dinounet_training.py:449)
INPLANE = 64                        # SPM conv_inplane (dinounet_training.py:757)
DEFORM_HEADS, DEFORM_POINTS = 16, 4
N_PREFIX = 5                        # cls + 4 storage tokens


# ----------------------------------------------------------------------------- parameter spec
def param_spec(model: str, num_classes: int = 2) -> List[Tuple[str, Tuple[int, ...], str]]:
    """(key, shape, kind) for every *unique* tensor of the reference state dict."""
    v = VARIANTS[model]
    D = v.dim
    out: List[Tuple[str, Tuple[int, ...], str]] = []
    A = "encoder.dinov3_adapter."
    Bk = A + "backbone."

    def lin(p, o, i, bias=True):
        out.append((p + ".weight", (o, i), "w"))
        if bias:
            out.append((p + ".bias", (o,), "b"))

    def norm(p, c):
        out.append((p + ".weight", (c,), "nw"))
        out.append((p + ".bias", (c,), "nb"))

    def bn(p, c):
        norm(p, c)
        out.append((p + ".running_mean", (c,), "rm"))
        out.append((p + ".running_var", (c,), "rv"))
        out.append((p + ".num_batches_tracked", (), "nbt"))

    def conv(p, o, i, k, bias=True, groups=1):
        out.append((p + ".weight", (o, i // groups, k, k), "w"))
        if bias:
            out.append((p + ".bias", (o,), "b"))

    def convT(p, i, o, bias=True):
        out.append((p + ".weight", (i, o, 2, 2), "wT"))
        if bias:
            out.append((p + ".bias", (o,), "b"))

    out.append((A + "level_embed", (3, D), "tok"))
    out.append((Bk + "cls_token", (1, 1, D), "tok"))
    out.append((Bk + "storage_tokens", (1, 4, D), "tok"))
    out.append((Bk + "mask_token", (1, D), "zero"))
    conv(Bk + "patch_embed.proj", D, 3, 16)
    out.append((Bk + "rope_embed.periods", (D // v.heads // 4,), "periods"))
    for i in range(v.depth):
        p = f"{Bk}blocks.{i}."
        norm(p + "norm1", D)
        lin(p + "attn.qkv", 3 * D, D, v.qkv_bias)
        if v.qkv_bias:
            out.append((p + "attn.qkv.bias_mask", (3 * D,), "bias_mask"))
        lin(p + "attn.proj", D, D)
        out.append((p + "ls1.gamma", (D,), "ls"))
        norm(p + "norm2", D)
        if v.ffn == "mlp":
            lin(p + "mlp.fc1", v.ffn_hidden, D)
            lin(p + "mlp.fc2", D, v.ffn_hidden)
        else:
            lin(p + "mlp.w1", v.ffn_hidden, D)
            lin(p + "mlp.w2", v.ffn_hidden, D)
            lin(p + "mlp.w3", D, v.ffn_hidden)
        out.append((p + "ls2.gamma", (D,), "ls"))
    norm(Bk + "norm", D)
    if v.local_cls_norm:
        norm(Bk + "local_cls_norm", D)
    # SPM
    S = A + "spm."
    conv(S + "stem.0", INPLANE, 3, 3, False); bn(S + "stem.1", INPLANE)
    conv(S + "stem.3", INPLANE, INPLANE, 3, False); bn(S + "stem.4", INPLANE)
    conv(S + "stem.6", INPLANE, INPLANE, 3, False); bn(S + "stem.7", INPLANE)
    conv(S + "conv2.0", 2 * INPLANE, INPLANE, 3, False); bn(S + "conv2.1", 2 * INPLANE)
    conv(S + "conv3.0", 4 * INPLANE, 2 * INPLANE, 3, False); bn(S + "conv3.1", 4 * INPLANE)
    conv(S + "conv4.0", 4 * INPLANE, 4 * INPLANE, 3, False); bn(S + "conv4.1", 4 * INPLANE)
    conv(S + "fc1", D, INPLANE, 1); conv(S + "fc2", D, 2 * INPLANE, 1)
    conv(S + "fc3", D, 4 * INPLANE, 1); conv(S + "fc4", D, 4 * INPLANE, 1)

    def extractor(p):
        norm(p + "query_norm", D); norm(p + "feat_norm", D)
        out.append((p + "attn.sampling_offsets.weight", (DEFORM_HEADS * DEFORM_POINTS * 2, D), "w_off"))
        out.append((p + "attn.sampling_offsets.bias", (DEFORM_HEADS * DEFORM_POINTS * 2,), "b_off"))
        lin(p + "attn.attention_weights", DEFORM_HEADS * DEFORM_POINTS, D)
        lin(p + "attn.value_proj", D // 2, D)
        lin(p + "attn.output_proj", D, D // 2)
        lin(p + "ffn.fc1", D // 4, D)
        conv(p + "ffn.dwconv.dwconv", D // 4, D // 4, 3, True, groups=D // 4)
        lin(p + "ffn.fc2", D, D // 4)
        norm(p + "ffn_norm", D)

    for i in range(4):
        extractor(f"{A}interactions.{i}.extractor.")
        if i == 3:
            extractor(f"{A}interactions.3.extra_extractors.0.")
            extractor(f"{A}interactions.3.extra_extractors.1.")
    convT(A + "up", D, D)
    for i in range(1, 5):
        bn(f"{A}norm{i}", D)
    # FAPM
    Fp = "encoder.fapm."
    conv(Fp + "shared_basis", RANK, D, 1)
    for i in range(4):
        conv(f"{Fp}specific_bases.{i}", RANK, D, 1)
    for i in range(4):
        conv(f"{Fp}film_generators.{i}", 2 * RANK, RANK, 1)
    for i, oc in enumerate(FEATURES):
        r = f"{Fp}refinement_blocks.{i}."
        conv(r + "0", oc, RANK, 1); norm(r + "1", oc)
        conv(r + "3.depthwise", oc, oc, 3, True, groups=oc)
        conv(r + "3.pointwise", oc, oc, 1); norm(r + "3.bn", oc)
        conv(r + "4", oc, oc, 1)
        red = max(1, oc // 16)
        conv(r + "5.fc.0", red, oc, 1); conv(r + "5.fc.2", oc, red, 1)
    for i, oc in enumerate(FEATURES):
        if oc != RANK:
            conv(f"{Fp}shortcut_projections.{i}", oc, RANK, 1)
    for i, oc in enumerate(FEATURES):
        convT(f"encoder.ups.{i}.up2", oc, oc)
    # decoder
    for s in range(3):
        below, skip = FEATURES[3 - s], FEATURES[2 - s]
        st = f"decoder.stages.{s}.convs."
        conv(st + "0.conv", skip, 2 * skip, 3); norm(st + "0.norm", skip)
        conv(st + "1.conv", skip, skip, 3); norm(st + "1.norm", skip)
    for s in range(3):
        convT(f"decoder.transpconvs.{s}", FEATURES[3 - s], FEATURES[2 - s])
    for s in range(3):
        conv(f"decoder.seg_layers.{s}", num_classes, FEATURES[2 - s], 1)
    return out


def expand_aliases(sd: Dict[str, Tensor]) -> Dict[str, Tensor]:
    """Add the duplicated keys of the reference state dict (SURVEY.md §3d):
    `decoder.encoder.*` == `encoder.*` and `...convs.N.all_modules.{0,1}` == `.conv/.norm`."""
    full = dict(sd)
    for k, t in sd.items():
        if k.startswith("decoder.stages.") and (".conv." in k or ".norm." in k):
            full[k.replace(".conv.", ".all_modules.0.").replace(".norm.", ".all_modules.1.")] = t
    for k, t in list(full.items()):
        if k.startswith("encoder."):
            full["decoder." + k] = t
    return full


def make_state_dict(model: str, num_classes: int = 2, seed: int = 0, aliases: bool = True) -> Dict[str, Tensor]:
    """Deterministic 'meaningful' random weights (SURVEY.md §0 facts 5-6): every transformer /
    deformable-attention path carries signal (LayerScale O(1), non-zero offset/attention projections,
    non-trivial BN running stats, bias_mask = [1,0,1]).  Each tensor has its own CPU generator seeded by
    (seed, crc32(key)), so the same dict is regenerated on any machine with the same torch."""
    v = VARIANTS[model]
    sd: Dict[str, Tensor] = {}
    for key, shape, kind in param_spec(model, num_classes):
        g = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
        rn = lambda *s: torch.randn(*s, generator=g, dtype=torch.float32)
        ru = lambda lo, hi, *s: torch.rand(*s, generator=g, dtype=torch.float32) * (hi - lo) + lo
        if kind == "w":
            fan_in = math.prod(shape[1:])
            t = rn(*shape) * (1.0 / math.sqrt(fan_in))
        elif kind == "wT":      # ConvTranspose2d [Cin, Cout, 2, 2]: each output pixel sums over Cin
            t = rn(*shape) * (1.0 / math.sqrt(shape[0]))
        elif kind == "w_off":   # offsets in pixels of the 32x32 value map: ~N(0,1) px on top of the bias grid
            t = rn(*shape) * (1.0 / math.sqrt(shape[1]))
        elif kind == "b_off":   # MSDeformAttn._reset_parameters grid init (ms_deform_attn.py:137-149)
            th = torch.arange(DEFORM_HEADS, dtype=torch.float32) * (2.0 * math.pi / DEFORM_HEADS)
            gi = torch.stack([th.cos(), th.sin()], -1)
            gi = (gi / gi.abs().max(-1, keepdim=True)[0]).view(DEFORM_HEADS, 1, 1, 2).repeat(1, 1, DEFORM_POINTS, 1)
            for i in range(DEFORM_POINTS):
                gi[:, :, i, :] *= i + 1
            t = gi.reshape(-1).clone()
        elif kind == "b":
            t = rn(*shape) * 0.05
        elif kind == "nw":
            t = ru(0.8, 1.2, *shape)
        elif kind == "nb":
            t = rn(*shape) * 0.1
        elif kind == "rm":
            t = rn(*shape) * 0.1
        elif kind == "rv":
            t = ru(0.5, 1.5, *shape)
        elif kind == "nbt":
            t = torch.zeros((), dtype=torch.int64)
        elif kind == "ls":
            t = ru(0.25, 0.75, *shape)
        elif kind == "tok":
            t = rn(*shape) * 0.5
        elif kind == "zero":
            t = torch.zeros(*shape)
        elif kind == "bias_mask":
            D = shape[0] // 3
            t = torch.cat([torch.ones(D), torch.zeros(D), torch.ones(D)])
        elif kind == "periods":  # rope_position_encoding.py:108-114 (base 100)
            d4 = shape[0]
            t = 100.0 ** (2 * torch.arange(d4, dtype=torch.float32) / (2 * d4))
        else:
            raise KeyError(kind)
        assert tuple(t.shape) == tuple(shape), (key, t.shape, shape)
        sd[key] = t
    return expand_aliases(sd) if aliases else sd


def make_input(batch: int, size: int, seed: int = 0, channels: int = 3) -> Tensor:
    g = torch.Generator().manual_seed(1234567 + seed)
    return torch.randn(batch, channels, size, size, generator=g, dtype=torch.float32)


# ----------------------------------------------------------------------------- forward pieces
def _ln(x, P, p, eps):
    return F.layer_norm(x, (x.shape[-1],), P[p + ".weight"], P[p + ".bias"], eps)


def _lin(x, P, p):
    return F.linear(x, P[p + ".weight"], P.get(p + ".bias"))


def _conv(x, P, p, stride=1, padding=0, groups=1):
    return F.conv2d(x, P[p + ".weight"], P.get(p + ".bias"), stride=stride, padding=padding, groups=groups)


def _bn(x, P, p):
    return F.batch_norm(x, P[p + ".running_mean"], P[p + ".running_var"], P[p + ".weight"], P[p + ".bias"],
                        False, 0.1, 1e-5)


def _inorm(x, P, p):
    return F.instance_norm(x, None, None, P[p + ".weight"], P[p + ".bias"], True, 0.1, 1e-5)


def rope_sincos(periods: Tensor, H: int, W: int) -> Tuple[Tensor, Tensor]:
    """rope_position_encoding.py:57-106, eval mode, normalize_coords='separate', fp32."""
    dd = dict(device=periods.device, dtype=torch.float32)
    ch = torch.arange(0.5, H, **dd) / H
    cw = torch.arange(0.5, W, **dd) / W
    coords = torch.stack(torch.meshgrid(ch, cw, indexing="ij"), dim=-1).flatten(0, 1)
    coords = 2.0 * coords - 1.0
    ang = 2 * math.pi * coords[:, :, None] / periods[None, None, :]
    ang = ang.flatten(1, 2).tile(2)
    return torch.sin(ang), torch.cos(ang)


def _rope(t: Tensor, sin: Tensor, cos: Tensor) -> Tensor:
    """attention.py:16-27,66-85: rotate the last (N - prefix) rows in fp32, cast back."""
    dt = t.dtype
    t = t.to(sin.dtype)
    prefix = t.shape[-2] - sin.shape[-2]
    body = t[:, :, prefix:, :]
    x1, x2 = body.chunk(2, dim=-1)
    body = body * cos + torch.cat([-x2, x1], dim=-1) * sin
    return torch.cat((t[:, :, :prefix, :], body), dim=-2).to(dt)


def vit_taps(P: Dict[str, Tensor], v: VariantCfg, x: Tensor, collect: Optional[dict] = None):
    """vision_transformer.py:265-318 with n=taps, norm=True, return_class_token=True."""
    Bk = "encoder.dinov3_adapter.backbone."
    B = x.shape[0]
    D, nh = v.dim, v.heads
    t = _conv(x, P, Bk + "patch_embed.proj", stride=16)
    h, w = t.shape[2], t.shape[3]
    t = t.flatten(2).transpose(1, 2)
    cls = P[Bk + "cls_token"] + 0 * P[Bk + "mask_token"]
    tok = torch.cat([cls.expand(B, -1, -1), P[Bk + "storage_tokens"].expand(B, -1, -1), t], dim=1)
    sin, cos = rope_sincos(P[Bk + "rope_embed.periods"], h, w)
    taps = []
    for i in range(v.depth):
        p = f"{Bk}blocks.{i}."
        y = _ln(tok, P, p + "norm1", 1e-5)
        bias = P[p + "attn.qkv.bias"] * P[p + "attn.qkv.bias_mask"].to(P[p + "attn.qkv.bias"].dtype) \
            if v.qkv_bias else None
        qkv = F.linear(y, P[p + "attn.qkv.weight"], bias)
        N = qkv.shape[1]
        q, k, val = torch.unbind(qkv.reshape(B, N, 3, nh, D // nh), 2)
        q, k, val = [z.transpose(1, 2) for z in (q, k, val)]
        q, k = _rope(q, sin, cos), _rope(k, sin, cos)
        a = F.scaled_dot_product_attention(q, k, val).transpose(1, 2).reshape(B, N, D)
        tok = tok + _lin(a, P, p + "attn.proj") * P[p + "ls1.gamma"]
        y = _ln(tok, P, p + "norm2", 1e-5)
        if v.ffn == "mlp":
            m = _lin(F.gelu(_lin(y, P, p + "mlp.fc1")), P, p + "mlp.fc2")
        else:
            m = _lin(F.silu(_lin(y, P, p + "mlp.w1")) * _lin(y, P, p + "mlp.w2"), P, p + "mlp.w3")
        tok = tok + m * P[p + "ls2.gamma"]
        if i in v.taps:
            o = _ln(tok, P, Bk + "norm", 1e-5)
            taps.append((o[:, N_PREFIX:], o[:, 0]))
            if collect is not None:
                collect[f"vit_tap{len(taps) - 1}"] = o[:, N_PREFIX:]
    return taps, (h, w)


def reference_points(shapes, device) -> Tensor:
    """dinov3_adapter.py:40-53."""
    pts = []
    for (H_, W_) in shapes:
        ry, rx = torch.meshgrid(torch.linspace(0.5, H_ - 0.5, H_, dtype=torch.float32, device=device),
                                torch.linspace(0.5, W_ - 0.5, W_, dtype=torch.float32, device=device),
                                indexing="ij")
        pts.append(torch.stack((rx.reshape(-1)[None] / W_, ry.reshape(-1)[None] / H_), -1))
    return torch.cat(pts, 1)[:, :, None]


def msda_core(value: Tensor, shapes, loc: Tensor, attw: Tensor) -> Tensor:
    """ms_deform_attn.py:71-92 (grid_sample formulation; == ops/src/cuda/ms_deform_im2col_cuda.cuh:242-304)."""
    N_, S_, M_, D_ = value.shape
    _, Lq_, _, L_, P_, _ = loc.shape
    vals = value.split([H_ * W_ for H_, W_ in shapes], dim=1)
    grids = 2 * loc - 1
    sampled = []
    for lid, (H_, W_) in enumerate(shapes):
        vl = vals[lid].flatten(2).transpose(1, 2).reshape(N_ * M_, D_, H_, W_)
        gl = grids[:, :, :, lid].transpose(1, 2).flatten(0, 1)
        sampled.append(F.grid_sample(vl, gl, mode="bilinear", padding_mode="zeros", align_corners=False))
    attw = attw.transpose(1, 2).reshape(N_ * M_, 1, Lq_, L_ * P_)
    out = (torch.stack(sampled, dim=-2).flatten(-2) * attw).sum(-1).view(N_, M_ * D_, Lq_)
    return out.transpose(1, 2).contiguous()


def msda_module(P, p, query, ref, feat, hw) -> Tensor:
    """MSDeformAttn.forward, ms_deform_attn.py:158-216 (n_levels=1, 16 heads, 4 points, ratio 0.5)."""
    N, Lq, _ = query.shape
    Hh, Ww = hw
    value = _lin(feat, P, p + "value_proj")
    value = value.view(N, feat.shape[1], DEFORM_HEADS, value.shape[-1] // DEFORM_HEADS)
    off = _lin(query, P, p + "sampling_offsets").view(N, Lq, DEFORM_HEADS, 1, DEFORM_POINTS, 2)
    aw = _lin(query, P, p + "attention_weights").view(N, Lq, DEFORM_HEADS, DEFORM_POINTS)
    aw = F.softmax(aw, -1).view(N, Lq, DEFORM_HEADS, 1, DEFORM_POINTS)
    normalizer = torch.tensor([[Ww, Hh]], dtype=torch.long, device=query.device)
    loc = ref[:, :, None, :, None, :] + off / normalizer[None, None, None, :, None, :]
    # custom_fwd(cast_inputs=float32): sampling runs in fp32 with autocast disabled (ms_deform_attn.py:30)
    with torch.autocast(device_type=query.device.type, enabled=False):
        o = msda_core(value.float(), [(Hh, Ww)], loc.float(), aw.float())
    return _lin(o, P, p + "output_proj")


def conv_ffn(P, p, x, H, W) -> Tensor:
    """ConvFFN/DWConv, dinov3_adapter.py:84-109."""
    x = _lin(x, P, p + "fc1")
    B, N, C = x.shape
    n = N // 21
    parts = []
    for sl, (hh, ww) in ((slice(0, 16 * n), (2 * H, 2 * W)), (slice(16 * n, 20 * n), (H, W)),
                         (slice(20 * n, N), (H // 2, W // 2))):
        t = x[:, sl, :].transpose(1, 2).reshape(B, C, hh, ww).contiguous()
        t = _conv(t, P, p + "dwconv.dwconv", padding=1, groups=C)
        parts.append(t.flatten(2).transpose(1, 2))
    x = F.gelu(torch.cat(parts, dim=1))
    return _lin(x, P, p + "fc2")


def extractor(P, p, c, ref, feat, hw_tok, H_c, W_c) -> Tensor:
    """Extractor.forward, dinov3_adapter.py:140-156 (eval: DropPath = identity; LN eps 1e-6)."""
    a = msda_module(P, p + "attn.", _ln(c, P, p + "query_norm", 1e-6), ref, _ln(feat, P, p + "feat_norm", 1e-6), hw_tok)
    c = c + a
    return c + conv_ffn(P, p + "ffn.", _ln(c, P, p + "ffn_norm", 1e-6), H_c, W_c)


def spm(P, x) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """SpatialPriorModule.forward, dinov3_adapter.py:279-302."""
    S = "encoder.dinov3_adapter.spm."
    c1 = F.relu(_bn(_conv(x, P, S + "stem.0", 2, 1), P, S + "stem.1"))
    c1 = F.relu(_bn(_conv(c1, P, S + "stem.3", 1, 1), P, S + "stem.4"))
    c1 = F.relu(_bn(_conv(c1, P, S + "stem.6", 1, 1), P, S + "stem.7"))
    c1 = F.max_pool2d(c1, 3, 2, 1)
    c2 = F.relu(_bn(_conv(c1, P, S + "conv2.0", 2, 1), P, S + "conv2.1"))
    c3 = F.relu(_bn(_conv(c2, P, S + "conv3.0", 2, 1), P, S + "conv3.1"))
    c4 = F.relu(_bn(_conv(c3, P, S + "conv4.0", 2, 1), P, S + "conv4.1"))
    c1, c2, c3, c4 = (_conv(c, P, S + f"fc{i + 1}") for i, c in enumerate((c1, c2, c3, c4)))
    tm = lambda t: t.flatten(2).transpose(1, 2)
    return c1, tm(c2), tm(c3), tm(c4)


def adapter_forward(P, v: VariantCfg, x: Tensor, autocast_like_reference: bool, collect=None) -> List[Tensor]:
    """DINOv3_Adapter.forward, dinov3_adapter.py:408-484 -> [f1, f2, f3, f4]."""
    A = "encoder.dinov3_adapter."
    bs, _, h, w = x.shape
    ref = reference_points([(h // 8, w // 8), (h // 16, w // 16), (h // 32, w // 32)], x.device)
    c1, c2, c3, c4 = spm(P, x)
    le = P[A + "level_embed"]
    c2, c3, c4 = c2 + le[0], c3 + le[1], c4 + le[2]
    n2, n3 = c2.shape[1], c3.shape[1]
    c = torch.cat([c2, c3, c4], dim=1)
    H_c, W_c = h // 16, w // 16
    with torch.autocast(device_type=x.device.type, dtype=torch.bfloat16,
                        enabled=autocast_like_reference and x.device.type == "cuda"):
        with torch.no_grad():
            taps, (Ht, Wt) = vit_taps(P, v, x, collect)
    outs = []
    for i in range(4):
        xi, _cls = taps[i]
        c = extractor(P, f"{A}interactions.{i}.extractor.", c, ref, xi, (Ht, Wt), H_c, W_c)
        if i == 3:
            for j in range(2):
                c = extractor(P, f"{A}interactions.3.extra_extractors.{j}.", c, ref, xi, (Ht, Wt), H_c, W_c)
        outs.append(xi.transpose(1, 2).reshape(bs, v.dim, Ht, Wt).contiguous())
        if collect is not None:
            collect[f"c_after{i}"] = c
    sp = lambda t, hh, ww: t.transpose(1, 2).reshape(bs, v.dim, hh, ww).contiguous()
    c2 = sp(c[:, :n2], H_c * 2, W_c * 2)
    c3 = sp(c[:, n2:n2 + n3], H_c, W_c)
    c4 = sp(c[:, n2 + n3:], H_c // 2, W_c // 2)
    c1 = F.conv_transpose2d(c2, P[A + "up.weight"], P[A + "up.bias"], stride=2) + c1
    sizes = [(4 * H_c, 4 * W_c), (2 * H_c, 2 * W_c), (H_c, W_c), (H_c // 2, W_c // 2)]
    xs = [F.interpolate(o, size=s, mode="bilinear", align_corners=False) for o, s in zip(outs, sizes)]
    cs = [c1 + xs[0], c2 + xs[1], c3 + xs[2], c4 + xs[3]]
    return [_bn(ci, P, f"{A}norm{i + 1}") for i, ci in enumerate(cs)]


def fapm_forward(P, feats: List[Tensor]) -> List[Tensor]:
    """FAPM.forward, dinounet_training.py:419-441."""
    Fp = "encoder.fapm."
    outs = []
    for i, x in enumerate(feats):
        zs = _conv(x, P, Fp + "shared_basis")
        zp = _conv(x, P, f"{Fp}specific_bases.{i}")
        gamma, beta = torch.chunk(_conv(zs, P, f"{Fp}film_generators.{i}"), 2, dim=1)
        z = gamma * zp + beta
        r = f"{Fp}refinement_blocks.{i}."
        t = F.leaky_relu(_inorm(_conv(z, P, r + "0"), P, r + "1"), 0.01)
        t = _conv(t, P, r + "3.depthwise", padding=1, groups=t.shape[1])
        t = F.leaky_relu(_inorm(_conv(t, P, r + "3.pointwise"), P, r + "3.bn"), 0.01)
        t = _conv(t, P, r + "4")
        wgt = torch.sigmoid(_conv(F.relu(_conv(F.adaptive_avg_pool2d(t, 1), P, r + "5.fc.0")), P, r + "5.fc.2"))
        t = t * wgt
        sc = _conv(z, P, f"{Fp}shortcut_projections.{i}") if (f"{Fp}shortcut_projections.{i}.weight" in P) else z
        outs.append(t + sc)
    return outs


def encoder_forward(P, v: VariantCfg, x: Tensor, autocast_like_reference=False, collect=None) -> List[Tensor]:
    """DINOv3EncoderAdapter.forward, dinounet_training.py:489-511."""
    B, C, H, W = x.shape
    if C == 1:
        x = x.repeat(1, 3, 1, 1)
    elif C != 3:
        x = x.repeat(1, 3 // C + (1 if 3 % C != 0 else 0), 1, 1)[:, :3] if C < 3 else x[:, :3]
    feats = adapter_forward(P, v, x, autocast_like_reference, collect)
    if collect is not None:
        for i, f in enumerate(feats):
            collect[f"f{i + 1}"] = f
    ys = fapm_forward(P, feats)
    skips = []
    for i, y in enumerate(ys):
        target = (H // (2 ** i), W // (2 ** i))
        hh, ww = y.shape[2], y.shape[3]
        while hh * 2 <= target[0] and ww * 2 <= target[1]:
            y = F.conv_transpose2d(y, P[f"encoder.ups.{i}.up2.weight"], P[f"encoder.ups.{i}.up2.bias"], stride=2)
            hh, ww = y.shape[2], y.shape[3]
        if (hh, ww) != target:
            y = F.interpolate(y, size=target, mode="bilinear", align_corners=False)
        skips.append(y)
        if collect is not None:
            collect[f"skip{i}"] = y
    return skips


def decoder_forward(P, skips: List[Tensor], collect=None) -> Tensor:
    """UNetDecoder.forward (deep_supervision=False), dinounet_training.py:603-629."""
    lres = skips[-1]
    for s in range(3):
        x = F.conv_transpose2d(lres, P[f"decoder.transpconvs.{s}.weight"], P[f"decoder.transpconvs.{s}.bias"], stride=2)
        x = torch.cat((x, skips[-(s + 2)]), 1)
        for j in range(2):
            p = f"decoder.stages.{s}.convs.{j}."
            x = F.leaky_relu(_inorm(_conv(x, P, p + "conv", 1, 1), P, p + "norm"), 0.01)
        lres = x
        if collect is not None:
            collect[f"dec{s}"] = x
    return _conv(lres, P, "decoder.seg_layers.2")


def forward(P: Dict[str, Tensor], model: str, x: Tensor, autocast_like_reference: bool = False,
            collect: Optional[dict] = None) -> Tensor:
    """DinoUNet.forward (dinounet_training.py:786-804).  With `autocast_like_reference=True` on a CUDA
    device this reproduces the reference's GPU precision regime: outer fp16 autocast (nnUNetTrainer.py:914,
    predict_from_raw_data.py:695), inner bf16 autocast around the frozen ViT (dinov3_adapter.py:422),
    fp32 deformable sampling (ms_deform_attn.py:30).  On CPU everything is fp32 (autocast('cuda') is inert)."""
    v = VARIANTS[model]
    with torch.no_grad():
        with torch.autocast(device_type=x.device.type, dtype=torch.float16,
                            enabled=autocast_like_reference and x.device.type == "cuda"):
            skips = encoder_forward(P, v, x, autocast_like_reference, collect)
            return decoder_forward(P, skips, collect)


def algorithmic_flops_per_patch(model: str, size: int = 512, num_classes: int = 2) -> float:
    """2*MAC forward FLOPs per patch (SURVEY.md §8d formulae), used by bench.py's roofline."""
    v = VARIANTS[model]
    D = v.dim
    P = (size // 16) ** 2
    N = P + N_PREFIX
    Lq = 21 * (size // 32) ** 2
    per_layer = 2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D
    per_layer += (4 if v.ffn == "mlp" else 6) * N * D * v.ffn_hidden
    fl = v.depth * per_layer + 2 * P * 768 * D
    s4, s8, s16, s32 = (size // 4) ** 2, (size // 8) ** 2, (size // 16) ** 2, (size // 32) ** 2
    fl += 2 * ((size // 2) ** 2 * (27 * 64 + 2 * 576 * 64) + s8 * 576 * 128 + s16 * 1152 * 256 + s32 * 2304 * 256)
    fl += 2 * D * (s4 * 64 + s8 * 128 + s16 * 256 + s32 * 256)
    ext = 2 * P * D * (D // 2) + 2 * Lq * D * (128 + 64) + 2 * Lq * (D // 2) * D + Lq * (D // 2) * 4 * 2 * 4 \
        + 4 * Lq * D * (D // 4) + 2 * Lq * (D // 4) * 9
    fl += 6 * ext
    fl += 2 * s8 * D * 4 * D
    for i, oc in enumerate(FEATURES):
        px = (size // (4 * 2 ** i)) ** 2
        fl += 2 * px * (2 * D * RANK + RANK * 2 * RANK + RANK * oc + 9 * oc + 2 * oc * oc + (RANK * oc if oc != RANK else 0))
        fl += 2 * px * oc * 4 * oc + 2 * 4 * px * oc * 4 * oc
    for s in range(3):
        below, skip = FEATURES[3 - s], FEATURES[2 - s]
        px_lo = (size // (8 // 2 ** s)) ** 2
        px_hi = 4 * px_lo
        fl += 2 * px_lo * below * 4 * skip + 2 * px_hi * 9 * (2 * skip * skip + skip * skip)
    fl += 2 * size * size * FEATURES[0] * num_classes
    return float(fl)
