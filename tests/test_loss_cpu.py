"""Loss oracle (oracle/loss_oracle.py) pinned against the REAL reference loss classes, through their answers stored in
tests/golden/ref_pins_loss.npz (oracle/make_golden_reference_pins.py), and against committed known answers; product-side
argument handling that needs no GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import loss_oracle as LO
from oracle.make_golden_reference_pins import LOSS_CASES, loss_case

PINS = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_pins_loss.npz"))


@pytest.mark.parametrize("batch_dice", [True, False])
def test_loss_oracle_equals_reference_classes(batch_dice):
    """DC_and_CE_loss(MemoryEfficientSoftDiceLoss) as nnUNetTrainer.py:363-365 builds it: loss and input gradient agree to
    fp32 reduction-order noise (bit-identical when computed on the same host; a vectorised sum's order depends on the
    host's SIMD width), the validation tp / fp / fn counts exactly."""
    for seed, (B, C) in enumerate(LOSS_CASES):
        z, t = loss_case(B, C, 24, 20, seed)
        z2 = z.clone().requires_grad_(True)
        got, _, _ = LO.dc_and_ce_loss(z2, t, batch_dice=batch_dice)
        got.backward()
        want = PINS[f"loss_bd{int(batch_dice)}_{seed}"]
        want_grad = PINS[f"grad_bd{int(batch_dice)}_{seed}"]
        assert abs(got.item() - float(want)) <= 1e-6 * max(1.0, abs(float(want)))
        assert np.abs(z2.grad.numpy() - want_grad).max() <= 1e-6 * np.abs(want_grad).max()
        tp, fp, fn = PINS[f"tp_fp_fn_{seed}"]
        otp, ofp, ofn = LO.validation_hard_counts(z, t)
        assert np.array_equal(otp.numpy(), tp) and np.array_equal(ofp.numpy(), fp) and np.array_equal(ofn.numpy(), fn)


def test_loss_oracle_known_answers():
    """Hand-checkable cases: a perfect confident prediction -> CE ~ 0, dice term ~ -1; uniform logits -> CE = ln C."""
    t = torch.zeros(1, 1, 4, 4)
    t[..., 2:] = 1
    z = torch.zeros(1, 2, 4, 4)
    z[:, 0] = torch.where(t[:, 0] == 0, 30.0, -30.0)
    z[:, 1] = -z[:, 0]
    loss, ce, dc = LO.dc_and_ce_loss(z, t)
    assert abs(float(ce)) < 1e-6 and abs(float(dc) + 1) < 1e-6 and abs(float(loss) + 1) < 1e-6
    loss, ce, dc = LO.dc_and_ce_loss(torch.zeros(2, 4, 8, 8), torch.zeros(2, 1, 8, 8))
    assert abs(float(ce) - np.log(4)) < 1e-6
    # no foreground at all: every fg class has I=0, G=0, P=N/4 -> dc_c = s / (P + s)
    assert abs(float(dc) + 1e-5 / (2 * 64 / 4 + 1e-5)) < 1e-9
    tp, fp, fn = LO.validation_hard_counts(z, t)
    assert tp.tolist() == [8, 8] and fp.tolist() == [0, 0] and fn.tolist() == [0, 0]


def test_product_loss_argument_contract():
    from dinounet_b200.loss import DC_and_CE_loss
    from dinounet_b200.lib import NativeLibraryError
    with pytest.raises(NotImplementedError):
        DC_and_CE_loss({"batch_dice": True}, {}, ignore_label=3)
    m = DC_and_CE_loss({"batch_dice": True, "smooth": 1e-5, "do_bg": False, "ddp": False}, {}, weight_ce=1, weight_dice=1)
    assert m.batch_dice and not m.do_bg and m.smooth == 1e-5
    with pytest.raises(NativeLibraryError):
        m(torch.zeros(1, 2, 4, 4), torch.zeros(1, 1, 4, 4))      # CPU tensors: no fallback
