"""TEST INFRASTRUCTURE — writes tests/golden/ref_pins_*.npz: the REAL reference's answers for the cases on which the CPU
tests pin the oracle restatements (forward, loss, gradients, sliding-window loop), so those tests run without the
reference.  Run where the reference sources are present (oracle/ref_loader.py):
    python oracle/make_golden_reference_pins.py
Inputs and weights are not stored: the tests regenerate them from the same seeds (CPU torch RNG).

  ref_pins_forward.npz         state-dict key -> shape of the reference module per model, and its fp32 logits for
                               tests/test_oracle_vs_reference.py (FORWARD_CASES + the single-channel input path)
  ref_pins_loss.npz            DC_and_CE_loss value + input gradient, and get_tp_fp_fn_tn counts (tests/test_loss_cpu.py)
  ref_pins_grads.npz           loss and per-parameter gradient statistics of autograd through the reference module
                               (tests/test_grad_oracle_cpu.py): names, absmax, L2 norm and a strided sample per tensor
  ref_pins_sliding_window.npz  fp16 result of nnUNetPredictor's sliding-window loop (tests/test_sliding_window_cpu.py)
"""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import dinounet_oracle as O  # noqa: E402
from oracle import loss_oracle as LO  # noqa: E402
from oracle.ref_loader import build_reference_model, load_reference_module  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# tests/test_oracle_vs_reference.py: weights seed 3, input (2, 3, size, size) seed 5
FORWARD_CASES = [("dinounet_s", 128), ("dinounet_b", 64), ("dinounet_7b_tiny", 64)]
# tests/test_loss_cpu.py: (B, C) per seed, logits (B, C, 24, 20)
LOSS_CASES = [(2, 2), (3, 4), (1, 3)]
# tests/test_grad_oracle_cpu.py: model, batch, size, classes, seed
GRAD_CASE = ("dinounet_s", 1, 128, 2, 3)
GRAD_SAMPLES = 64
# tests/test_sliding_window_cpu.py: (c, H, W) image, patch, step, gaussian, mirror axes; seed = 5 + index, 3 heads
SW_CASES = [((3, 2, 70, 45), (32, 32), 0.5, True, (0, 1)), ((1, 1, 100, 100), (64, 64), 0.3, True, (0,))]


def loss_case(B, C, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C, H, W, generator=g) * 3, torch.randint(0, C, (B, 1, H, W), generator=g).float()


def grad_case(model, B, S, ncls, seed):
    sd = O.make_state_dict(model, ncls, seed=seed)
    x = O.make_input(B, S, seed)
    target = torch.randint(0, ncls, (B, 1, S, S), generator=torch.Generator().manual_seed(seed + 7)).float()
    return sd, x, target


def strided_sample(t: torch.Tensor, n: int = GRAD_SAMPLES) -> torch.Tensor:
    f = t.reshape(-1)
    return f[:: max(1, f.numel() // n)][:n]


def forward_pins():
    out = {}
    for model, size in FORWARD_CASES:
        sd = O.make_state_dict(model, 2, seed=3)
        net = build_reference_model(model, 2)
        out[f"keys_{model}"] = np.array(json.dumps({k: list(t.shape) for k, t in net.state_dict().items()}))
        net.load_state_dict(sd, strict=True)
        with torch.no_grad():
            out[f"logits_{model}_s{size}"] = net(O.make_input(2, size, 5)).numpy()
    sd = O.make_state_dict("dinounet_s", 2, seed=3)
    net = build_reference_model("dinounet_s", 2, sd)
    with torch.no_grad():
        out["logits_single_channel"] = net(O.make_input(1, 64, 7, channels=1)).numpy()
    return out


def loss_pins():
    DC_and_CE_loss, MemDice, get_tp_fp_fn_tn = LO.load_reference_loss()
    out = {}
    for batch_dice in (True, False):
        ref = DC_and_CE_loss({"batch_dice": batch_dice, "smooth": 1e-5, "do_bg": False, "ddp": False}, {}, weight_ce=1,
                             weight_dice=1, ignore_label=None, dice_class=MemDice)          # nnUNetTrainer.py:363-365
        for seed, (B, C) in enumerate(LOSS_CASES):
            z, t = loss_case(B, C, 24, 20, seed)
            z = z.requires_grad_(True)
            loss = ref(z, t)
            loss.backward()
            out[f"loss_bd{int(batch_dice)}_{seed}"] = loss.detach().numpy()
            out[f"grad_bd{int(batch_dice)}_{seed}"] = z.grad.numpy()
    for seed, (B, C) in enumerate(LOSS_CASES):
        z, t = loss_case(B, C, 24, 20, seed)
        pred = torch.zeros_like(z).scatter_(1, z.argmax(1)[:, None], 1)
        tp, fp, fn, _ = get_tp_fp_fn_tn(pred, t, axes=[0, 2, 3], mask=None)
        out[f"tp_fp_fn_{seed}"] = torch.stack([tp, fp, fn]).numpy()
    return out


def grad_pins():
    model, B, S, ncls, seed = GRAD_CASE
    sd, x, target = grad_case(model, B, S, ncls, seed)
    net = build_reference_model(model, ncls, sd)          # eval mode: BN running stats, DropPath off
    load_reference_module()
    msda_mod = sys.modules["dinounet.dinov3.eval.segmentation.models.utils.ms_deform_attn"]

    class _Differentiable:                                 # the extension-backed backward cannot run on CPU
        @staticmethod
        def apply(value, shapes, lsi, loc, aw, step):
            return msda_mod.ms_deform_attn_core_pytorch(value, shapes, loc, aw)

    orig = msda_mod.MSDeformAttnFunction
    msda_mod.MSDeformAttnFunction = _Differentiable
    try:
        DC_and_CE_loss, MemDice, _ = LO.load_reference_loss()
        crit = DC_and_CE_loss({"batch_dice": True, "smooth": 1e-5, "do_bg": False, "ddp": False}, {}, weight_ce=1,
                              weight_dice=1, ignore_label=None, dice_class=MemDice)
        loss = crit(net(x), target)
        loss.backward()
    finally:
        msda_mod.MSDeformAttnFunction = orig
    # the reference's named_parameters() lists each shared Parameter once
    grads = {n: p.grad for n, p in sorted(net.named_parameters()) if p.requires_grad}
    names = sorted(grads)
    none = [n for n in names if grads[n] is None]
    live = [n for n in names if grads[n] is not None]
    return {"loss": np.float64(loss.item()), "names": np.array(names), "none": np.array(none, dtype=str),
            "live": np.array(live), "absmax": np.array([grads[n].abs().max().item() for n in live], dtype=np.float64),
            "norm": np.array([grads[n].double().norm().item() for n in live]),
            "samples": np.stack([np.pad(strided_sample(grads[n]).numpy(), (0, GRAD_SAMPLES))[:GRAD_SAMPLES] for n in live]),
            "n_samples": np.array([strided_sample(grads[n]).numel() for n in live])}


def sliding_window_pins():
    from oracle.make_golden_sliding_window import reference_loop
    out = {}
    for k, (shape, patch, step, ug, ma) in enumerate(SW_CASES):
        _, y = reference_loop(shape, patch, step, ug, ma, heads=3, seed=k + 5)
        out[f"loop_{k}"] = y.numpy()
    return out


def main():
    for name, fn in (("forward", forward_pins), ("loss", loss_pins), ("grads", grad_pins),
                     ("sliding_window", sliding_window_pins)):
        with contextlib.redirect_stdout(io.StringIO()):
            arrays = fn()
        path = os.path.join(GOLDEN, f"ref_pins_{name}.npz")
        np.savez_compressed(path, **arrays)
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
