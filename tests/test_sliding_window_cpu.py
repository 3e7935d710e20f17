"""Sliding-window predictor, CPU side: the oracle restatement against the golden vectors produced by the REAL reference
(`oracle/make_golden_sliding_window.py`, `oracle/make_golden_reference_pins.py`), and the product's host-side
functions (steps, gaussian, padding, slicers, mirror order) against both."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import sliding_window_oracle as SWO
from oracle.make_golden_reference_pins import SW_CASES
from dinounet_b200 import sliding_window as SW

KAT = np.load(os.path.join(os.path.dirname(__file__), "golden", "sliding_window_kat.npz"))
LOOP_CASES = [((1, 2, 40, 56), (32, 32), 0.5, True, (0, 1)), ((3, 1, 20, 70), (32, 32), 0.5, True, (0, 1)),
              ((2, 3, 64, 33), (32, 32), 0.25, False, None), ((4, 1, 50, 50), (32, 32), 0.5, True, (1,))]


def toy_network(cin, heads, seed=0):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(heads, cin, 3, 3, generator=g) * 0.5
    b = torch.randn(heads, generator=g)
    return lambda x: torch.nn.functional.conv2d(x.float(), w, b, padding=1).half()


def test_steps_match_reference_golden():
    for image, tile, step, want in json.loads(bytes(KAT["steps_json"]).decode()):
        assert SWO.compute_steps_for_sliding_window(image, tile, step) == want
        assert SW.compute_steps_for_sliding_window(image, tile, step) == want
    with pytest.raises(AssertionError):
        SW.compute_steps_for_sliding_window((100,), (64,), 0.0)


def test_gaussian_matches_reference_golden_bitwise():
    cpu = torch.device("cpu")
    for n in (32, 512):
        want = KAT[f"gaussian_{n}"]
        for fn in (SWO.compute_gaussian, SW.compute_gaussian):
            got = fn((n, n), sigma_scale=1. / 8, value_scaling_factor=10, device=cpu).numpy()
            assert got.dtype == np.float16 and np.array_equal(got, want)
    want = KAT["gaussian_48x20_scale1"]
    assert np.array_equal(SWO.compute_gaussian((48, 20), device=cpu).numpy(), want)
    assert np.array_equal(SW.compute_gaussian((48, 20), device=cpu).numpy(), want)
    assert (want > 0).all()


def test_gaussian_restatement_equals_scipy_filter():
    from scipy.ndimage import gaussian_filter
    for size in ((32, 32), (17, 64), (512, 512)):
        tmp = np.zeros(size)
        tmp[tuple(i // 2 for i in size)] = 1
        want = gaussian_filter(tmp, [i / 8 for i in size], 0, mode="constant", cval=0)
        got = SWO.compute_gaussian(size, dtype=torch.float64).numpy()
        assert np.array_equal(got, want / want.max())


@pytest.mark.parametrize("case", range(len(LOOP_CASES)))
def test_oracle_loop_matches_reference_golden_bitwise(case):
    shape, patch, step, ug, ma = LOOP_CASES[case]
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(1))
    y = SWO.predict_sliding_window_return_logits(toy_network(shape[0], 2), x, patch, 2, step, ug, ma)
    assert y.dtype == torch.half and np.array_equal(y.numpy(), KAT[f"loop_{case}"])


def test_oracle_loop_matches_live_reference_predictor():
    """nnUNetPredictor.predict_sliding_window_return_logits around a 3-head toy network, as run by
    oracle/make_golden_reference_pins.py (input seeded like reference_loop's: seed + 1)."""
    pins = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_pins_sliding_window.npz"))
    for k, (shape, patch, step, ug, ma) in enumerate(SW_CASES):
        seed = k + 5
        x = torch.randn(*shape, generator=torch.Generator().manual_seed(seed + 1))
        got = SWO.predict_sliding_window_return_logits(toy_network(shape[0], 3, seed), x, patch, 3, step, ug, ma)
        assert got.dtype == torch.half and np.array_equal(got.numpy(), pins[f"loop_{k}"])


def test_product_padding_slicers_and_mirror_order():
    x = torch.arange(2 * 3 * 20 * 70, dtype=torch.float32).reshape(2, 3, 20, 70)
    a, sa = SWO.pad_nd_image(x, (32, 32))
    b, sb = SW.pad_to_patch_size(x, (32, 32))
    assert torch.equal(a, b) and sa == sb and a.shape == (2, 3, 32, 70) and torch.equal(a[sa], x)
    c, sc = SW.pad_to_patch_size(x, (16, 16))
    assert c is x and sc == tuple(slice(0, s) for s in x.shape)

    p = SW.SlidingWindowPredictor.__new__(SW.SlidingWindowPredictor)        # host logic only: no device needed
    p.configuration_manager = SimpleNamespace(patch_size=[32, 32])
    p.tile_step_size, p.verbose = 0.5, False
    assert p._internal_get_sliding_window_slicers((3, 64, 90)) == SWO.get_sliding_window_slicers((3, 64, 90), [32, 32], 0.5)
    p.use_mirroring, p.allowed_mirroring_axes = True, (0, 1)
    assert p._mirror_variants() == [0, 1, 2, 3]            # none, dim 2, dim 3, both (predict_from_raw_data.py:545-550)
    p.allowed_mirroring_axes = (1,)
    assert p._mirror_variants() == [0, 2]
    p.use_mirroring = False
    assert p._mirror_variants() == [0]


def test_product_predictor_refuses_cpu():
    from dinounet_b200.lib import NativeLibraryError
    with pytest.raises(NativeLibraryError):
        SW.SlidingWindowPredictor(device=torch.device("cpu"))
