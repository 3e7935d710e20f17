"""CPU: the oracle restatement against the REAL reference forward, through the reference's answers stored in
tests/golden/ref_pins_forward.npz (oracle/make_golden_reference_pins.py, same seeds): the state-dict keys and shapes must
match exactly; the logits agree to fp32 reduction-order noise.  Run on the same host with the same thread count the two
are bit-identical; the stored logits are compared within 2e-5 abs, because the host's thread count alone moves the
oracle's last bits by up to ~7e-6 (1 vs 8 threads; the same bound as tests/test_oracle_golden.py)."""
import json
import os

import numpy as np
import pytest

from oracle import dinounet_oracle as O

PINS = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_pins_forward.npz"))
TOL = 2e-5


def _check(y, ref):
    assert y.shape == ref.shape
    assert np.abs(y - ref).max() <= TOL
    margin = np.abs(ref[:, 0] - ref[:, 1])
    assert ((y.argmax(1) != ref.argmax(1)) & (margin > 1e-4)).sum() == 0


@pytest.mark.parametrize("model,size", [("dinounet_s", 128), ("dinounet_b", 64), ("dinounet_7b_tiny", 64)])
def test_bit_identical_to_reference(model, size):
    sd = O.make_state_dict(model, 2, seed=3)
    ref_shapes = json.loads(str(PINS[f"keys_{model}"]))
    assert set(ref_shapes) == set(sd)
    for k, shape in ref_shapes.items():
        assert list(sd[k].shape) == shape, k
    x = O.make_input(2, size, 5)
    _check(O.forward(sd, model, x).numpy(), PINS[f"logits_{model}_s{size}"])


def test_single_channel_input_path():
    """dinounet_training.py:491-497 channel fix-up."""
    sd = O.make_state_dict("dinounet_s", 2, seed=3)
    x = O.make_input(1, 64, 7, channels=1)
    _check(O.forward(sd, "dinounet_s", x).numpy(), PINS["logits_single_channel"])
