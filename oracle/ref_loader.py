"""TEST INFRASTRUCTURE ONLY — imports the REAL reference (the original DinoUNet sources, at
$DINOUNET_REFERENCE_ROOT) on CPU.

Used by the golden generators (`oracle/make_golden.py`, `oracle/make_golden_reference_pins.py`) to pin the oracle
restatement (`oracle/dinounet_oracle.py`) against the reference's own forward; the tests compare with what those
generators stored under tests/golden/ and never need the reference itself.

Shims (SURVEY.md §8c):
  1. `dinounet/__init__.py` pulls `api.py` -> batchgenerators (absent): pre-seed
     `sys.modules['dinounet']` as a bare namespace package and stub `dinounet.api` and
     `dinounet.training.nnUNetTrainer.nnUNetTrainerNoDeepSupervision`
     (dinounet_training.py:7-8).
  2. `dynamic_network_architectures` (requirements.txt:3, absent): stand-ins for the 5
     symbols imported at dinounet_training.py:13-20, restating the published semantics of
     dynamic-network-architectures 0.4.x (`ConvDropoutNormReLU`, `StackedConvBlocks`).
  3. `MultiScaleDeformableAttention` (ms_deform_attn.py:18 imports it unconditionally):
     a stub module; the live forward never calls it (it uses grid_sample).
  4. `pretrained=False` is forced (no network): `load_dinov3_model` is patched.
"""
import importlib
import os
import sys
import types

import torch
from torch import nn

REF_ROOT = os.environ.get("DINOUNET_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "dinounet_training.py"))


class _ConvDropoutNormReLU(nn.Module):
    """dynamic_network_architectures.building_blocks.simple_conv_blocks.ConvDropoutNormReLU (0.4.x)."""

    def __init__(self, conv_op, input_channels, output_channels, kernel_size, stride, conv_bias=False,
                 norm_op=None, norm_op_kwargs=None, dropout_op=None, dropout_op_kwargs=None,
                 nonlin=None, nonlin_kwargs=None, nonlin_first=False):
        super().__init__()
        if not isinstance(kernel_size, (tuple, list)):
            kernel_size = [kernel_size] * 2
        if not isinstance(stride, (tuple, list)):
            stride = [stride] * 2
        norm_op_kwargs = norm_op_kwargs or {}
        nonlin_kwargs = nonlin_kwargs or {}
        ops = []
        self.conv = conv_op(input_channels, output_channels, kernel_size, stride,
                            padding=[(i - 1) // 2 for i in kernel_size], dilation=1, bias=conv_bias)
        ops.append(self.conv)
        if dropout_op is not None:
            self.dropout = dropout_op(**dropout_op_kwargs)
            ops.append(self.dropout)
        if norm_op is not None:
            self.norm = norm_op(output_channels, **norm_op_kwargs)
            ops.append(self.norm)
        if nonlin is not None:
            self.nonlin = nonlin(**nonlin_kwargs)
            ops.append(self.nonlin)
        if nonlin_first and (norm_op is not None and nonlin is not None):
            ops[-1], ops[-2] = ops[-2], ops[-1]
        self.all_modules = nn.Sequential(*ops)

    def forward(self, x):
        return self.all_modules(x)


class _StackedConvBlocks(nn.Module):
    """dynamic_network_architectures...simple_conv_blocks.StackedConvBlocks (0.4.x)."""

    def __init__(self, num_convs, conv_op, input_channels, output_channels, kernel_size, initial_stride,
                 conv_bias=False, norm_op=None, norm_op_kwargs=None, dropout_op=None, dropout_op_kwargs=None,
                 nonlin=None, nonlin_kwargs=None, nonlin_first=False):
        super().__init__()
        if not isinstance(output_channels, (tuple, list)):
            output_channels = [output_channels] * num_convs
        args = (conv_bias, norm_op, norm_op_kwargs, dropout_op, dropout_op_kwargs, nonlin, nonlin_kwargs, nonlin_first)
        self.convs = nn.Sequential(
            _ConvDropoutNormReLU(conv_op, input_channels, output_channels[0], kernel_size, initial_stride, *args),
            *[_ConvDropoutNormReLU(conv_op, output_channels[i - 1], output_channels[i], kernel_size, 1, *args)
              for i in range(1, num_convs)])
        self.output_channels = output_channels[-1]

    def forward(self, x):
        return self.convs(x)


def _install_shims():
    if "dinounet_training" in sys.modules:
        return
    if not reference_available():
        raise RuntimeError(f"reference not present at {REF_ROOT}")

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    # (1) bare namespace for `dinounet`
    pkg = mod("dinounet")
    pkg.__path__ = [os.path.join(REF_ROOT, "dinounet")]
    mod("dinounet.api", plan_and_preprocess=None, training=None, evaluate=None)
    tr = mod("dinounet.training"); tr.__path__ = []
    nt = mod("dinounet.training.nnUNetTrainer"); nt.__path__ = []

    class nnUNetTrainerNoDeepSupervision:  # stub base class
        pass

    mod("dinounet.training.nnUNetTrainer.nnUNetTrainerNoDeepSupervision",
        nnUNetTrainerNoDeepSupervision=nnUNetTrainerNoDeepSupervision)

    # (2) dynamic_network_architectures stand-ins
    d = mod("dynamic_network_architectures"); d.__path__ = []
    bb = mod("dynamic_network_architectures.building_blocks"); bb.__path__ = []

    def convert_conv_op_to_dim(conv_op):
        return {nn.Conv1d: 1, nn.Conv2d: 2, nn.Conv3d: 3}[conv_op]

    def get_matching_convtransp(conv_op=None, dimension=None):
        return {nn.Conv1d: nn.ConvTranspose1d, nn.Conv2d: nn.ConvTranspose2d, nn.Conv3d: nn.ConvTranspose3d}[conv_op]

    mod("dynamic_network_architectures.building_blocks.helper",
        convert_conv_op_to_dim=convert_conv_op_to_dim, get_matching_convtransp=get_matching_convtransp)
    mod("dynamic_network_architectures.building_blocks.plain_conv_encoder", PlainConvEncoder=nn.Module)
    mod("dynamic_network_architectures.building_blocks.simple_conv_blocks",
        StackedConvBlocks=_StackedConvBlocks, ConvDropoutNormReLU=_ConvDropoutNormReLU)
    ini = mod("dynamic_network_architectures.initialization"); ini.__path__ = []

    class InitWeights_He:
        def __init__(self, neg_slope=1e-2):
            self.neg_slope = neg_slope

        def __call__(self, module):
            pass

    mod("dynamic_network_architectures.initialization.weight_init", InitWeights_He=InitWeights_He)

    # (3) native extension stub (forward never calls it)
    if "MultiScaleDeformableAttention" not in sys.modules:
        mod("MultiScaleDeformableAttention")

    sys.path.insert(0, REF_ROOT)
    importlib.import_module("dinounet_training")


def load_reference_module():
    """Returns the imported (unmodified) `dinounet_training` module of the reference."""
    _install_shims()
    return sys.modules["dinounet_training"]


PLANS_ARCH = {
    # what the planner emits for main_dinov3's forced 2d/512/4-stage plan (SURVEY.md §8 row A0)
    "n_stages": 4,
    "features_per_stage": [32, 64, 128, 256],
    "conv_op": "torch.nn.modules.conv.Conv2d",
    "kernel_sizes": [[3, 3]] * 4,
    "strides": [[1, 1], [2, 2], [2, 2], [2, 2]],
    "n_conv_per_stage": [2, 2, 2, 2],
    "n_conv_per_stage_decoder": [2, 2, 2],
    "conv_bias": True,
    "norm_op": "torch.nn.modules.instancenorm.InstanceNorm2d",
    "norm_op_kwargs": {"eps": 1e-5, "affine": True},
    "dropout_op": None,
    "dropout_op_kwargs": None,
    "nonlin": "torch.nn.LeakyReLU",
    "nonlin_kwargs": {"inplace": True},
}


def _register_tiny_7b(ref):
    """Adds the test-only `dinounet_7b_tiny` recipe (dinov3_vit7b16's kwargs, hub/backbones.py:452-494, at small size) to
    the reference's own registries so the REAL reference code builds it."""
    if "dinounet_7b_tiny" in ref.DINOv3_MODEL_FACTORIES:
        return
    from dinounet.dinov3.hub.backbones import _make_dinov3_vit

    def factory(*, pretrained=False, **kw):
        return _make_dinov3_vit(img_size=224, patch_size=16, in_chans=3, pos_embed_rope_base=100,
                                pos_embed_rope_normalize_coords="separate", pos_embed_rope_rescale_coords=2,
                                pos_embed_rope_dtype="fp32", embed_dim=1024, depth=4, num_heads=8, ffn_ratio=3,
                                qkv_bias=False, drop_path_rate=0.4, layerscale_init=1.0e-05, norm_layer="layernormbf16",
                                ffn_layer="swiglu64", ffn_bias=True, proj_bias=True, n_storage_tokens=4, mask_k_bias=True,
                                untie_global_and_local_cls_norm=True, pretrained=False, compact_arch_name="vit7b")

    ref.DINOv3_MODEL_FACTORIES["dinounet_7b_tiny"] = factory
    ref.DINOv3_INTERACTION_INDEXES["dinounet_7b_tiny"] = [0, 1, 2, 3]
    ref.DINOv3_MODEL_INFO["dinounet_7b_tiny"] = {"embed_dim": 1024, "depth": 4, "num_heads": 8, "params": "test"}


def build_reference_model(model_name: str, num_classes: int = 2, state_dict=None):
    """Build the REAL reference DinoUNet (random-init, no download) in eval mode on CPU."""
    ref = load_reference_module()
    _register_tiny_7b(ref)

    def _load_no_download(name, pretrained_path=None):
        return ref.DINOv3_MODEL_FACTORIES[name](pretrained=False)

    orig = ref.load_dinov3_model
    ref.load_dinov3_model = _load_no_download
    try:
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            net = ref.DinoUNet.from_config({"architecture": dict(PLANS_ARCH)}, 3, num_classes,
                                           dinov3_pretrained_path=None, dinov3_model_name=model_name)
    finally:
        ref.load_dinov3_model = orig
    if state_dict is not None:
        net.load_state_dict(state_dict, strict=True)
    return net.eval()
