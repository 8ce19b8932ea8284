"""The tolerance model of test_conv_layers_gpu.py, on the CPU.

A float64 emulation of a bf16x3 layer (value + residual bf16 operands, three products, exact accumulation) must pass the
per-layer bounds TOL_ELEM / TOL_RMS, and every emulation of a layer that lost part of its arithmetic must exceed both
bounds by SENS x -- otherwise the GPU test could not tell a correct kernel from a broken one.
"""
import pytest

from test_conv_layers_gpu import (BROKEN, SENS, TOL_ELEM, TOL_RMS, conv_op, emulate, fails_clearly, make_input, make_weights,
                                  passes, reference, rel_errors)

# (kind, stride, A, c_in, H, W, n_out): 3x3 stride 1 / 2 at the benched widths, a deep 256-channel layer, 1x1, deblock
LAYERS = [("conv3", 1, 2, 64, 16, 32, 64), ("conv3", 2, 2, 64, 17, 31, 64), ("conv3", 1, 2, 256, 8, 16, 64),
          ("conv1", 1, 2, 96, 16, 16, 48), ("deconv", 2, 2, 128, 8, 8, 32)]


def _layer(kind, stride, A, c_in, H, W, n_out):
    x = make_input(c_in + H, A, c_in, H, W)
    k = 3 if kind == "conv3" else 1 if kind == "conv1" else stride
    shape = (c_in, n_out, k, k) if kind == "deconv" else (n_out, c_in, k, k)
    w, b = make_weights(c_in + W, shape, c_in * (k * k if kind != "deconv" else 1), n_out)
    return conv_op(kind, stride), x, w, b, 0 if kind == "deconv" else 1


@pytest.mark.parametrize("layer", LAYERS, ids=lambda l: f"{l[0]}_s{l[1]}_{l[3]}to{l[6]}")
def test_bf16x3_emulation_passes_and_broken_ones_fail(layer):
    op, x, w, b, in_dim = _layer(*layer)
    ref, absc = reference(op, x, w, b)
    good = rel_errors(emulate(op, x, w, b, "bf16x3", in_dim=in_dim), ref, absc)
    assert passes(good), good
    # the margin the GPU bounds leave a correct layer
    assert good[0] * SENS <= TOL_ELEM and good[1] * SENS <= TOL_RMS, good
    for mode in BROKEN:
        bad = rel_errors(emulate(op, x, w, b, mode, in_dim=in_dim), ref, absc)
        assert fails_clearly(bad), (mode, bad, (SENS * TOL_ELEM, SENS * TOL_RMS))


def test_heads_emulation_without_activation():
    """The detection heads have a bias but no ReLU: negative outputs count too."""
    op = conv_op("conv1")
    x = make_input(7, 2, 256, 8, 16)
    w, b = make_weights(8, (20, 256, 1, 1), 256, 20)
    ref, absc = reference(op, x, w, b, relu=False)
    assert passes(rel_errors(emulate(op, x, w, b, "bf16x3", relu=False), ref, absc))
    assert fails_clearly(rel_errors(emulate(op, x, w, b, "act_residual_dropped", relu=False), ref, absc))


def test_error_measure():
    """Where absconv is 0 the reference is exactly 0: any deviation there is an unbounded relative error."""
    import torch
    ref, absc = torch.zeros(4, dtype=torch.float64), torch.tensor([0.0, 1.0, 1.0, 0.0], dtype=torch.float64)
    assert rel_errors(torch.zeros(4), ref + 0, absc)[0] == 0.0
    assert rel_errors(torch.tensor([0.0, 0.0, 0.0, 1e-30]), ref, absc)[0] == float("inf")
