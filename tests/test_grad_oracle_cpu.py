"""Gradient oracle (oracle/grad_oracle.py = autograd through the oracle forward + loss oracle), the round-2 backward
target: pinned against autograd through the REAL reference module + REAL reference loss (stored in
tests/golden/ref_pins_grads.npz), and against committed golden gradient norms / samples of the oracle itself."""
import glob
import os

import numpy as np
import torch

from oracle import dinounet_oracle as O
from oracle import grad_oracle as G
from oracle.make_golden_reference_pins import GRAD_CASE, strided_sample


def _case(model, B, S, ncls, seed):
    sd = O.make_state_dict(model, ncls, seed=seed)
    x = O.make_input(B, S, seed)
    target = torch.randint(0, ncls, (B, 1, S, S), generator=torch.Generator().manual_seed(seed + 7)).float()
    return sd, x, target


def test_grad_oracle_matches_golden():
    files = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "grads_*.npz")))
    assert files
    for f in files:
        model, b, s, c, w = os.path.basename(f)[len("grads_"):-4].rsplit("_", 4)
        g = np.load(f)
        sd, x, target = _case(model, int(b[1:]), int(s[1:]), int(c[1:]), int(w[1:]))
        loss, grads = G.loss_and_grads(sd, model, x, target)
        assert abs(loss.item() - float(g["loss"])) < 1e-6
        names = [str(n) for n in g["names"]]
        assert names == sorted(grads)
        norms = np.array([grads[k].double().norm().item() for k in names])
        # the conv biases ahead of an InstanceNorm have an exactly zero true gradient: their stored norms (below 1e-6 of
        # the largest) are fp32 rounding noise that differs from host to host, so those only have to stay that small
        floor = 1e-6 * g["norms"].max()
        zero = g["norms"] < floor
        assert (norms[zero] < floor).all(), [n for n, z, v in zip(names, zero, norms) if z and v >= floor]
        assert np.allclose(norms[~zero], g["norms"][~zero], rtol=1e-4, atol=1e-9), \
            [(n, v, w) for n, v, w in zip(names, norms, g["norms"]) if w >= floor and not np.isclose(v, w, rtol=1e-4, atol=1e-9)]
        for i, k in enumerate(names):
            fl = grads[k].reshape(-1)
            samp = fl[:: max(1, fl.numel() // 16)][:16].numpy()
            assert np.allclose(samp, g[f"s{i}"], rtol=1e-3, atol=1e-7), k


def test_grad_oracle_equals_reference_autograd():
    """Against autograd through the reference module + reference loss (MSDA core swapped for its differentiable
    pure-PyTorch twin, the extension's backward being CUDA-only), stored by oracle/make_golden_reference_pins.py: the loss,
    the trainable-parameter set, and per tensor the absmax, the L2 norm and a strided sample of the gradient, each within
    1e-4 of the tensor's scale.  The conv biases ahead of an InstanceNorm have an exactly zero true gradient; what
    autograd leaves there (below 1e-6 of the largest gradient) is fp32 rounding noise that moves with the host's thread
    count, so for those tensors the oracle's gradient must be as small, not equal."""
    pins = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_pins_grads.npz"))
    model, B, S, ncls, seed = GRAD_CASE
    sd, x, target = _case(model, B, S, ncls, seed)
    loss, grads = G.loss_and_grads(sd, model, x, target)
    assert abs(loss.item() - float(pins["loss"])) < 1e-6
    # the reference's named_parameters() lists each shared Parameter once; every trainable oracle key must be among them
    names = {str(n) for n in pins["names"]}
    assert names == set(grads), (sorted(names ^ set(grads))[:10])
    for k in pins["none"]:
        assert float(grads[str(k)].abs().max()) == 0.0, k
    floor = 1e-6 * float(pins["absmax"].max())
    worst = 0.0
    for i, k in enumerate(str(n) for n in pins["live"]):
        go, amax, norm = grads[k], float(pins["absmax"][i]), float(pins["norm"][i])
        if amax <= floor:
            assert float(go.abs().max()) <= floor, k
            continue
        samp = strided_sample(go).numpy()
        n = int(pins["n_samples"][i])
        assert samp.size == n, k
        worst = max(worst, float(np.abs(samp - pins["samples"][i, :n]).max()) / amax,
                    abs(float(go.abs().max()) - amax) / amax, abs(go.double().norm().item() - norm) / norm)
    assert worst < 1e-4, worst
