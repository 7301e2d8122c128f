"""CPU tests: the oracles against the golden vectors generated from the reference module
(oracle/make_golden.py) plus analytic known-answer and property tests (SURVEY.md 4, 8c)."""
import glob
import os

import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

from cfdbench_b200 import synth
from oracle import fno_numpy as onp
from oracle import fno_torch_port as opt

from conftest import GOLDEN

CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))


def load_case(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    problem = str(g["problem"])
    p = synth.n_case_params(problem)
    sd = synth.make_state_dict(int(g["weight_seed"]), n_params=p, spectral_gain=float(g["spectral_gain"]))
    batch = synth.make_batch(int(g["batch_seed"]), g["preds"].shape[0], problem)
    return g, sd, batch


def test_golden_present():
    assert len(CASES) >= 3


@pytest.mark.parametrize("name", CASES)
def test_torch_port_matches_reference_golden(name):
    g, sd, batch = load_case(name)
    tb = {k: torch.from_numpy(v) for k, v in batch.items()}
    pp = opt.params_from_numpy(sd, requires_grad=True)
    out = opt.forward(pp, tb["inputs"], tb["case_params"], tb["mask"], tb["label"], return_acts=True)
    # same library calls as the reference: bit-exact on the generating host, 1e-6 elsewhere
    # (MKL/oneDNN thread partitioning may reorder sums)
    assert onp.rel_l2(out["preds"].detach().numpy(), g["preds"].astype(np.float64)) < 1e-6
    loss = np.array([out["loss"][k].item() for k in ("mse", "rmse", "mae", "nmse")])
    np.testing.assert_allclose(loss, g["loss"], rtol=1e-5)
    ch = g["act_channels"]   # the fixtures keep these hidden channels of each activation
    assert onp.rel_l2(out["acts"][0][:1, ch].detach().numpy(), g["act0_b0"].astype(np.float64)) < 1e-6
    assert onp.rel_l2(out["acts"][1][:1, ch].detach().numpy(), g["act1_b0"].astype(np.float64)) < 1e-6
    assert onp.rel_l2(out["acts"][-1][:1, ch].detach().numpy(), g["act4_b0"].astype(np.float64)) < 1e-6
    out["loss"]["nmse"].backward()
    for key in g.files:
        if key.startswith("grad::"):
            k = key[6:]
            ref = g[key]
            err = np.linalg.norm(pp[k].grad.numpy() - ref) / np.linalg.norm(ref)
            assert err < 1e-4, (k, err)
    steps = int(g["steps"])
    roll = opt.rollout(opt.params_from_numpy(sd), tb["inputs"], tb["case_params"], tb["mask"], steps)
    for s in range(steps):
        assert onp.rel_l2(roll[s].numpy(), g["rollout"][s].astype(np.float64)) < 1e-5, s


@pytest.mark.parametrize("name", CASES)
def test_numpy_oracle_matches_reference_golden(name):
    g, sd, batch = load_case(name)
    out = onp.fno_forward(sd, batch["inputs"], batch["case_params"], batch["mask"], batch["label"],
                          return_acts=True)
    ch = g["act_channels"]
    assert onp.rel_l2(g["preds"], out["preds"]) < 2e-6
    assert onp.rel_l2(g["act0_b0"], out["acts"][0][:1, ch]) < 2e-6
    assert onp.rel_l2(g["act1_b0"], out["acts"][1][:1, ch]) < 2e-6
    for i, k in enumerate(("mse", "rmse", "mae", "nmse")):
        assert abs(out["loss"][k] - g["loss"][i]) <= 2e-6 * abs(g["loss"][i])
    # the first spectral convolution, fed with the lift output checked just above
    spec = onp.spectral_conv(out["acts"][0][:1], sd["blocks.0.conv0.weights1"], sd["blocks.0.conv0.weights2"])
    assert onp.rel_l2(g["spectral0_b0"], spec[:, ch]) < 2e-6


def test_numpy_oracle_gradients_match_reference_golden():
    g, sd, batch = load_case("cylinder_b2_gain200")
    grads = onp.fno_backward(sd, batch["inputs"], batch["case_params"], batch["mask"], batch["label"])
    for key in g.files:
        if key.startswith("grad::"):
            k = key[6:]
            err = np.linalg.norm(grads[k] - g[key]) / np.linalg.norm(g[key])
            assert err < 5e-5, (k, err)
        elif key.startswith("gradslice::"):
            k = key[11:]
            sl = grads[k][:, :, ::4, ::4]
            err = np.linalg.norm(sl - g[key]) / np.linalg.norm(g[key])
            assert err < 5e-5, (k, err)
            assert abs(np.linalg.norm(grads[k]) - float(g["gradnorm::" + k])) < 5e-5 * float(g["gradnorm::" + k])


# ---------------------------------------------------------------------------------- known answers

def _one_hot_weights(i, o, kxi, ky, value, m=12, c=32):
    w = np.zeros((c, c, 2 * m, m), dtype=np.complex128)
    w[i, o, kxi, ky] = value
    return w[:, :, :m].astype(np.complex64), w[:, :, m:].astype(np.complex64)


@pytest.mark.parametrize("a,b_", [(3, 5), (0, 4), (7, 0), (-2, 3), (-11, 11)])
def test_single_mode_known_answer(a, b_):
    """x = cos(2 pi (a h + b w)/64) on channel i with a one-hot weight on mode (a,b) gives
    |g| cos(2 pi (a h + b w)/64 + arg g) * (1/2 or 1) on channel o and zero elsewhere."""
    h = np.arange(64)[:, None]
    w = np.arange(64)[None, :]
    x = np.zeros((1, 32, 64, 64))
    x[0, 4] = np.cos(2 * np.pi * (a * h + b_ * w) / 64)
    gval = complex(np.complex64(0.7 - 0.4j))  # weights are stored as complex64
    kxi = a if a >= 0 else 24 + a
    w1, w2 = _one_hot_weights(4, 9, kxi, b_, gval)
    y = onp.spectral_conv(x, w1, w2)
    # X[a,b] = 2048 (or 4096 if the mode is its own mirror); output keeps only the (a,b) half
    amp = 4096.0 if (a % 64 == 0 and b_ == 0) else 2048.0
    c = 1.0 if b_ == 0 else 2.0
    if b_ == 0 and a != 0:
        # ky = 0 column: the mirror row -a is not weighted, so only half the cosine survives
        expect = (amp / 4096.0) * np.real(gval * np.exp(2j * np.pi * (a * h + b_ * w) / 64))
    else:
        expect = c * (amp / 4096.0) * np.real(gval * np.exp(2j * np.pi * (a * h + b_ * w) / 64))
    np.testing.assert_allclose(y[0, 9], expect, atol=1e-9)
    others = np.delete(y[0], 9, axis=0)
    assert np.abs(others).max() < 1e-9
    # torch port agrees
    yt = opt.spectral_conv(torch.from_numpy(x.astype(np.float32)), torch.from_numpy(w1), torch.from_numpy(w2))
    np.testing.assert_allclose(yt.numpy()[0, 9], expect, atol=2e-5)


def test_dc_imaginary_part_is_dropped():
    """A purely imaginary product on mode (0,0) contributes nothing (C2R drops Im of ky=0 DC)."""
    x = np.ones((1, 32, 64, 64))
    w1, w2 = _one_hot_weights(0, 0, 0, 0, 1j)
    assert np.abs(onp.spectral_conv(x, w1, w2)).max() < 1e-12
    yt = opt.spectral_conv(torch.ones(1, 32, 64, 64), torch.from_numpy(w1), torch.from_numpy(w2))
    assert yt.abs().max().item() < 1e-6


def test_zero_spectral_weights_reduce_block_to_pointwise():
    sd = synth.make_state_dict(5)
    sd["blocks.0.conv0.weights1"][:] = 0
    sd["blocks.0.conv0.weights2"][:] = 0
    x = np.random.default_rng(0).standard_normal((1, 32, 64, 64))
    y = onp.fno_block(x, sd, 0)
    expect = onp.gelu(onp.conv1x1(x, sd["blocks.0.w0.weight"], sd["blocks.0.w0.bias"]))
    np.testing.assert_allclose(y, expect, atol=1e-12)


def test_numpy_oracle_equals_numpy_fft():
    """The truncated-DFT closed form equals numpy's own rfft2/irfft2 pipeline."""
    rng = np.random.default_rng(3)
    x = rng.standard_normal((2, 32, 64, 64))
    sd = synth.make_state_dict(9, spectral_gain=100.0)
    w1, w2 = sd["blocks.1.conv0.weights1"], sd["blocks.1.conv0.weights2"]
    xf = np.fft.rfft2(x)
    of = np.zeros((2, 32, 64, 33), dtype=np.complex128)
    of[:, :, :12, :12] = np.einsum("bixy,ioxy->boxy", xf[:, :, :12, :12], w1)
    of[:, :, -12:, :12] = np.einsum("bixy,ioxy->boxy", xf[:, :, -12:, :12], w2)
    ref = np.fft.irfft2(of, s=(64, 64))
    np.testing.assert_allclose(onp.spectral_conv(x, w1, w2), ref, atol=1e-10)


def test_spectral_adjoint_is_consistent():
    """<gy, J dx> == <J^T gy, dx> and finite-difference check of the weight gradient."""
    rng = np.random.default_rng(4)
    x = rng.standard_normal((1, 32, 64, 64))
    dx = rng.standard_normal((1, 32, 64, 64))
    gy = rng.standard_normal((1, 32, 64, 64))
    sd = synth.make_state_dict(10, spectral_gain=50.0)
    w1, w2 = sd["blocks.0.conv0.weights1"], sd["blocks.0.conv0.weights2"]
    gx, gw1, gw2 = onp.spectral_conv_backward(x, w1, w2, gy)
    lhs = np.sum(gy * onp.spectral_conv(dx, w1, w2))
    rhs = np.sum(gx * dx)
    assert abs(lhs - rhs) < 1e-9 * max(1.0, abs(lhs))
    dw = np.zeros_like(w1, dtype=np.complex128)
    dw[3, 7, 2, 5] = 1e-3 + 2e-3j
    f0 = np.sum(gy * onp.spectral_conv(x, w1, w2))
    f1 = np.sum(gy * onp.spectral_conv(x, (w1 + dw).astype(np.complex128), w2))
    pred = np.real(np.conj(gw1[3, 7, 2, 5]) * dw[3, 7, 2, 5])
    assert abs((f1 - f0) - pred) < 1e-6 * max(1.0, abs(pred))


@settings(max_examples=5, deadline=None)
@given(st.floats(-2, 2), st.floats(-2, 2), st.integers(0, 2**31 - 1))
def test_spectral_conv_is_linear(alpha, beta, seed):
    rng = np.random.default_rng(seed)
    x1 = rng.standard_normal((1, 32, 64, 64)).astype(np.float32)
    x2 = rng.standard_normal((1, 32, 64, 64)).astype(np.float32)
    sd = synth.make_state_dict(1, spectral_gain=100.0)
    w1 = torch.from_numpy(sd["blocks.0.conv0.weights1"])
    w2 = torch.from_numpy(sd["blocks.0.conv0.weights2"])
    f = lambda t: opt.spectral_conv(torch.from_numpy(t), w1, w2).numpy()
    lhs = f(alpha * x1 + beta * x2)
    rhs = alpha * f(x1) + beta * f(x2)
    assert np.abs(lhs - rhs).max() < 1e-4 * (1 + np.abs(rhs).max())


def test_bf16_boundary_oracle_error_budget():
    """SURVEY.md 7 precision contract: rounding hidden activations to bf16 costs ~2e-3 rel-L2."""
    sd = synth.make_state_dict(7)
    batch = synth.make_batch(8, 2, "cavity")
    tb = {k: torch.from_numpy(v) for k, v in batch.items()}
    p = opt.params_from_numpy(sd)
    a = opt.forward(p, tb["inputs"], tb["case_params"], tb["mask"])["preds"].numpy()
    b = opt.forward(p, tb["inputs"], tb["case_params"], tb["mask"], round_fn=opt.bf16_round)["preds"].numpy()
    e = onp.rel_l2(b, a.astype(np.float64))
    assert 1e-4 < e < 1e-2
