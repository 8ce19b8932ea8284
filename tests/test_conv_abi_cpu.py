"""Packed-weight and workspace sizes of the tcgen05 convolution layers (host-only C entries, no GPU).

Every packer and launcher takes the packed N from one rule (conv_n_pad in csrc/conv_layer.cuh): the smallest of 32 / 64 / 128 /
256 that holds n_out, at least 64 for gc_conv_pack / gc_conv_planes and at least 32 for the heads, DoubleConv and the Enhancer.
These sizes are what callers allocate, so they must not move: the expected values below are written out independently of
the library, and matched the library before the kernel selection moved into conv_layer.cu."""
import itertools

import pytest

from gencomm_b200 import _lib

TAPS = (1, 9)
C_IN = (32, 64, 96, 384)
N_OUT = (8, 20, 24, 48, 64, 80, 128, 200, 256)
SHIPPED_C = (64, 128, 256, 384)
GRIDS = ((64, 128), (128, 256), (63, 127), (1, 1))


def n_pad(n, n_min):
    n = max(n, n_min)
    return next(p for p in (32, 64, 128, 256) if n <= p)


def align(x):
    return (x + 255) // 256 * 256


def out_size(n, stride):
    return (n - 1) // stride + 1


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def test_conv_packed_bytes(lib):
    for taps, c_in, n in itertools.product(TAPS, C_IN, N_OUT):
        assert lib.gc_conv_packed_bytes(taps, c_in, n) == taps * c_in * n_pad(n, 64) * 4, (taps, c_in, n)
    assert lib.gc_conv_packed_bytes(3, 64, 64) == 0 and lib.gc_conv_packed_bytes(9, 0, 64) == 0
    assert lib.gc_conv_packed_bytes(9, 64, 0) == 0
    assert lib.gc_conv_packed_bytes(9, 64, 20) == 147456     # below 64 outputs: packed for N = 64


def test_det_heads_bytes(lib):
    for C, n in itertools.product(SHIPPED_C + C_IN, N_OUT):
        assert lib.gc_det_heads_packed_bytes(C, n) == C * n_pad(n, 32) * 4, (C, n)
    assert lib.gc_det_heads_packed_bytes(256, 20) == 32768   # the shipped heads: N = 32
    assert lib.gc_det_heads_packed_bytes(0, 20) == 0 and lib.gc_det_heads_packed_bytes(64, 0) == 0
    for (H, W), frames, C in itertools.product(GRIDS, (1, 8), SHIPPED_C):
        assert lib.gc_det_heads_workspace_bytes(frames, C, H, W) == 2 * align(frames * H * W * C * 2), (frames, C, H, W)
    assert lib.gc_det_heads_workspace_bytes(0, 256, 64, 128) == 0


def test_double_conv_bytes(lib):
    for c_in, c_out in itertools.product(C_IN + SHIPPED_C, N_OUT):
        n = n_pad(c_out, 32)
        assert lib.gc_double_conv_packed_bytes(c_in, c_out) == align(9 * c_in * n * 4) + 9 * c_out * n * 4, (c_in, c_out)
    assert lib.gc_double_conv_packed_bytes(384, 128) == 2359296      # GenComm stage 1 shrink header
    for (H, W), stride, A, c_in, c_out in itertools.product(GRIDS, (1, 2), (1, 5), C_IN, N_OUT):
        hw_out = out_size(H, stride) * out_size(W, stride)
        plane = A * 2 * max(c_in * H * W, c_out * hw_out)
        ws = 2 * align(plane) + align(A * c_out * hw_out * 4)
        assert lib.gc_double_conv_workspace_bytes(A, c_in, H, W, stride, c_out) == ws, (A, c_in, H, W, stride, c_out)
        assert lib.gc_double_conv_planes_workspace_bytes(A, H, W, stride, c_out) == align(A * c_out * hw_out * 4)
    assert lib.gc_double_conv_workspace_bytes(1, 64, 64, 128, 0, 64) == 0
    assert lib.gc_double_conv_planes_workspace_bytes(1, 64, 128, 2, 0) == 0


def test_enhancer_packed_bytes(lib):
    for C in SHIPPED_C + (512,):
        expect = 0
        if C % 128 == 0:   # [partial_conv3: N = C/4][linear1: C/64 chunks of N = 256][linear2: C/128 chunks of N = 128]
            expect = align(9 * (C // 4) * (C // 4) * 4) + (C // 64) * C * 256 * 4 + (C // 128) * 2 * C * 128 * 4
        assert lib.gc_enhancer_packed_bytes(C) == expect, C
    assert lib.gc_enhancer_packed_bytes(128) == 430080
