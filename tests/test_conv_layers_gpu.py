"""Every tcgen05 convolution path of gc_conv_planes / gc_det_heads, one layer at a time, against a float64 reference.

A case runs one layer through the C ABI with random folded weights and bias and checks, element by element and in
aggregate, how far the result is from ReLU(conv(x, w) + b) evaluated in float64 on the same fp32 inputs:

  * element-wise  |got - ref| <= TOL_ELEM * absconv,  absconv = conv(|x|, |w|) + |b|   (a wrong tap, pixel, agent, channel
    chunk or a stale tile is far outside this);
  * aggregate     ||got - ref||_2 / ||ref||_2 <= TOL_RMS                                    (a lost bf16x3 pass is outside it);
  * sensitivity   the same layer emulated in float64 with the activation residual dropped fails both bounds by SENS x,
    so the bounds can tell a correct kernel from one that lost a precision pass;
  * sentinel      outputs are pre-filled with NaN (fp32) / 0xFF bytes (planes): everything outside the output channel window
    keeps the fill bit for bit, everything inside is finite;
  * planes        a plane output equals the host-side value / residual split of the same layer's NCHW output bit for bit.

Which kernel ran is asserted from torch.profiler in a pass of its own.  The switches that the library reads once per process
(GC_CONV_TMA, GC_CONV_MC, GC_CONV_MT2) are exercised in child processes (this file's __main__), which must reproduce the
default path bit for bit.  The constants and host helpers here are shared with test_conv_tolerance_cpu.py, which checks the
tolerance model on the CPU.
"""
import json
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

if __name__ == "__main__":     # child process: the package is imported from the repository tree
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# Per-layer bounds, set from the B200 measurements of this file's cases (DESIGN.md 5e): correct layers reach max(d/absconv)
# 1.3e-5 (1x1, c_in = 32: the fewest products per output) and <= 7.7e-6 everywhere else, rms <= 8.6e-6; a layer without the
# activation residual reaches >= 3.3e-4 (256 -> 256 3x3 over 2 tiles: the deepest K, the fewest outputs) and rms >= 1.6e-3.
TOL_ELEM = 6.5e-5
TOL_RMS = 5e-5
SENS = 5.0        # a broken emulation must exceed both bounds by this factor

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ------------------------------------------------------------------------------------------------
# host helpers (device-agnostic; test_conv_tolerance_cpu.py runs them on the CPU)
# ------------------------------------------------------------------------------------------------
def bf16_split(v):
    """(value, residual) bf16 of fp32 v: round-to-nearest bf16 of v, then of v - float(value) (implicit_gemm.cuh
    bf16_residual; the fp32 subtraction is exact)."""
    hi = v.to(torch.bfloat16)
    return hi, (v - hi.float()).to(torch.bfloat16)


def make_input(seed, A, C, H, W):
    """[A, C, H, W] fp32 on the CPU: agent a drawn from its own seed and scaled by 1 + a / 4 (a tile written to the wrong
    agent shows), border rows and columns x4 (a halo / out-of-bounds fill mistake shows), ~30 % exact zeros."""
    x = torch.empty(A, C, H, W)
    for a in range(A):
        g = torch.Generator().manual_seed(seed * 1009 + a)
        v = torch.randn(C, H, W, generator=g) * (1.0 + a / 4.0)
        v[:, 0] *= 4.0
        v[:, -1] *= 4.0 if H > 1 else 1.0
        v[:, :, 0] *= 4.0
        v[:, :, -1] *= 4.0 if W > 1 else 1.0
        v[torch.rand(C, H, W, generator=g) < 0.3] = 0.0
        x[a] = v
    return x


def make_weights(seed, shape, fan_in, n_bias):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) / fan_in ** 0.5, 0.1 * torch.randn(n_bias, generator=g)


def conv_op(kind, stride=1):
    """float64 pre-activation of the layer: 3x3 (padding 1, stride 1 | 2), 1x1, or ConvTranspose2d with kernel == stride."""
    if kind == "conv3":
        return lambda x, w, b: F.conv2d(x, w, b, stride=stride, padding=1)
    if kind == "conv1":
        return lambda x, w, b: F.conv2d(x, w, b)
    return lambda x, w, b: F.conv_transpose2d(x, w, b, stride=stride)


def _act(y, relu):
    return torch.relu(y) if relu else y


def reference(op, x, w, b, relu=True):
    """(ReLU(op(x, w) + b), op(|x|, |w|) + |b|) in float64 on the fp32 inputs."""
    xd, wd, bd = x.double(), w.double(), b.double()
    return _act(op(xd, wd, bd), relu), op(xd.abs(), wd.abs(), bd.abs())


BROKEN = ("act_residual_dropped", "weight_residual_dropped", "bf16", "stage_missing")


def emulate(op, x, w, b, mode, relu=True, in_dim=1):
    """float64 emulation of the layer's arithmetic.  "bf16x3": hi*hi + lo*hi + hi*lo (the kernels' three MMAs, exact
    accumulation); the broken variants drop the activation residual (lo*hi), the weight residual (hi*lo), both (one bf16
    pass), or the first 32-channel stage of the centre tap.  in_dim: the input-channel dimension of w (1 for a conv,
    0 for a transposed conv)."""
    xh, xl = (t.double() for t in bf16_split(x))
    wh, wl = (t.double() for t in bf16_split(w))
    bd = b.double()
    z = torch.zeros_like(bd)
    if mode == "stage_missing":
        ky, kx = w.shape[2] // 2, w.shape[3] // 2
        keep = torch.ones_like(wh)
        keep.narrow(in_dim, 0, 32)[..., ky, kx] = 0.0
        wh, wl = wh * keep, wl * keep
    y = op(xh, wh, bd)
    if mode in ("bf16x3", "weight_residual_dropped", "stage_missing"):
        y = y + op(xl, wh, z)
    if mode in ("bf16x3", "act_residual_dropped", "stage_missing"):
        y = y + op(xh, wl, z)
    return _act(y, relu)


def rel_errors(got, ref, absc):
    """(max |got - ref| / absconv, ||got - ref||_2 / ||ref||_2); where absconv is 0 the reference is exactly 0 and so must
    be the result."""
    d = (got.double() - ref).abs()
    elem = torch.where(absc > 0, d / absc.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    return float(elem.max()), float(d.norm() / ref.norm().clamp_min(1e-300))


def passes(errs):
    return errs[0] <= TOL_ELEM and errs[1] <= TOL_RMS


def fails_clearly(errs):
    return errs[0] >= SENS * TOL_ELEM and errs[1] >= SENS * TOL_RMS


# ------------------------------------------------------------------------------------------------
# GPU plumbing
# ------------------------------------------------------------------------------------------------
NAN_BITS = 0x7FC00000          # torch's fp32 NaN fill
PLANE_FILL = 0xFF              # plane sentinel bytes (bf16 0xFFFF is a NaN)


def kernel_name(raw):
    """'void ct::k_conv_tma<64, 9, 5, (bool)0, (bool)1>(CUtensorMap_st, ...)' -> 'k_conv_tma<64,9,5,0,1>'."""
    s = raw.replace("(bool)", "").replace("true", "1").replace("false", "0")
    s = s[5:] if s.startswith("void ") else s
    s = s.split("(")[0].replace(" ", "")
    base, _, args = s.partition("<")
    return base.split("::")[-1] + ("<" + args if args else "")


def launched(fn):
    """(fn(), names of the project's kernels it launched, in order) from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    names = [kernel_name(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return r, [n for n in names if n.startswith("k_")]


def template_args(name):
    return name.partition("<")[2].rstrip(">").split(",")


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def host_planes(x):
    """x [A, C, H, W] fp32 -> (xh, xl) channel-last bf16 planes as uint8 blobs [A][H][W][C] (built on the host: any C)."""
    hi, lo = bf16_split(x.permute(0, 2, 3, 1).contiguous())
    return hi.view(torch.uint8).reshape(-1), lo.view(torch.uint8).reshape(-1)


def plane_view(blob, A, H, W, C):
    return blob.view(torch.bfloat16).view(A, H, W, C).permute(0, 3, 1, 2)      # [A, C, H, W] view of [A][H][W][C]


def check_sentinel_nchw(out, lo, hi):
    """Channels [lo, hi) finite, every other element still the NaN fill bit for bit."""
    bits = out.view(torch.int32)
    outside = torch.cat([bits[:, :lo].reshape(-1), bits[:, hi:].reshape(-1)])
    assert bool((outside == NAN_BITS).all()), "an element outside the output channel window was written"
    assert bool(torch.isfinite(out[:, lo:hi]).all()), "an element inside the output channel window is not finite / not written"


def check_sentinel_planes(buf, A, H, W, C, lo, hi):
    for p in range(2):
        v = buf[p].view(A, H * W, C, 2)
        outside = torch.cat([v[:, :, :lo].reshape(-1), v[:, :, hi:].reshape(-1)])
        assert bool((outside == PLANE_FILL).all()), "a plane element outside the output channel window was written"
        assert bool(torch.isfinite(plane_view(buf[p], A, H, W, C)[:, lo:hi].float()).all()), \
            "a plane element inside the output channel window is not finite / not written"


def decode_planes(buf, A, H, W, C, lo, hi):
    """float64 value + residual of channels [lo, hi) of [2][A][H][W][C] bf16 planes -> [A, hi - lo, H, W]."""
    return plane_view(buf[0], A, H, W, C)[:, lo:hi].double() + plane_view(buf[1], A, H, W, C)[:, lo:hi].double()


def assert_split_matches(nchw, buf, A, H, W, C, lo, hi, what):
    """The plane output equals the host-side value / residual split of the NCHW output bit for bit."""
    hi_ref, lo_ref = bf16_split(nchw[:, lo:hi])
    for p, ref in ((0, hi_ref), (1, lo_ref)):
        got = plane_view(buf[p], A, H, W, C)[:, lo:hi]
        neq = int((got.view(torch.int16) != ref.view(torch.int16)).sum())
        assert neq == 0, f"{what}: {'value' if p == 0 else 'residual'} plane differs from the split of the NCHW output at {neq} elements"


def _report(case, kind, kernels, errs, broken):
    print(f"\n  {case + '/' + kind:34s} {','.join(sorted(set(kernels))):44s} max(d/absconv) {errs[0]:.2e}  rms {errs[1]:.2e}"
          f"  | act-residual dropped: {broken[0]:.2e} {broken[1]:.2e}", end="")


def assert_layer(case, kind, kernels, got, ref, absc, broken_out):
    errs, broken = rel_errors(got, ref, absc), rel_errors(broken_out, ref, absc)
    _report(case, kind, kernels, errs, broken)
    assert fails_clearly(broken), (f"{case}/{kind}: the bounds ({TOL_ELEM:g}, {TOL_RMS:g}) do not reject a layer without the "
                                   f"activation residual ({broken[0]:.2e}, {broken[1]:.2e})")
    assert passes(errs), f"{case}/{kind}: max(d/absconv) {errs[0]:.3e} (<= {TOL_ELEM:g}), rms {errs[1]:.3e} (<= {TOL_RMS:g})"


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
class ConvCase:
    """One gc_conv_planes layer: ReLU(conv(x, w) + b), 3x3 (stride 1 | 2) or 1x1, written as planes and / or NCHW into
    channels [off, off + n_out) of a `total`-channel output.  expect: kind -> kernel names that must run."""

    def __init__(self, name, A, c_in, H, W, n_out, taps=9, stride=1, total=None, off=0, expect=None, kinds=None, many=False):
        self.name, self.A, self.c_in, self.H, self.W, self.n_out = name, A, c_in, H, W, n_out
        self.taps, self.stride, self.total, self.off = taps, stride, total or n_out, off
        self.Ho, self.Wo = ((H - 1) // stride + 1, (W - 1) // stride + 1) if taps == 9 else (H, W)
        self.kinds = kinds or (("planes", "nchw") if n_out % 16 == 0 else ("nchw",))
        self.expect = expect or {}
        self.many = many               # n_tiles >= 3 x SM count: the persistent loop reuses each TMEM accumulator set
        self.n_tiles = A * self.Ho * self.Wo // 128
        self.seed = sum(map(ord, name))

    def prepare(self, dev):
        k = 3 if self.taps == 9 else 1
        x = make_input(self.seed, self.A, self.c_in, self.H, self.W)
        w, b = make_weights(self.seed + 1, (self.n_out, self.c_in, k, k), self.c_in * k * k, self.n_out)
        from gencomm_b200 import ops
        x, w, b = x.to(dev), w.to(dev), b.to(dev)
        return {"x": x, "w": w, "b": b, "planes": host_planes(x), "packed": ops.conv_pack(w)}

    def launch(self, st, kind):
        from gencomm_b200 import ops
        A, Ho, Wo = self.A, self.Ho, self.Wo
        args = (st["planes"], A, self.c_in, self.H, self.W, st["packed"], st["b"], self.n_out, self.taps)
        if kind == "planes":
            out = torch.full((2, A * Ho * Wo * self.total * 2), PLANE_FILL, dtype=torch.uint8, device=st["x"].device)
            ops.conv_planes(*args, stride=self.stride, out_planes=(out[0], out[1]), out_ch_total=self.total, out_ch_off=self.off)
        else:
            out = torch.full((A, self.total, Ho, Wo), float("nan"), device=st["x"].device)
            ops.conv_planes(*args, stride=self.stride, out_nchw=out, out_ch_off=self.off)
        return out

    def decode(self, kind, out):
        lo, hi = self.off, self.off + self.n_out
        if kind == "planes":
            return decode_planes(out, self.A, self.Ho, self.Wo, self.total, lo, hi)
        return out[:, lo:hi].double()

    def sentinel(self, kind, out):
        lo, hi = self.off, self.off + self.n_out
        if kind == "planes":
            check_sentinel_planes(out, self.A, self.Ho, self.Wo, self.total, lo, hi)
        else:
            check_sentinel_nchw(out, lo, hi)

    def split_matches(self, nchw, planes):
        assert_split_matches(nchw, planes, self.A, self.Ho, self.Wo, self.total, self.off, self.off + self.n_out, self.name)

    def op(self):
        return conv_op("conv3" if self.taps == 9 else "conv1", self.stride)

    def check(self, st, kind, out, kernels):
        self.sentinel(kind, out)
        op = self.op()
        ref, absc = reference(op, st["x"], st["w"], st["b"])
        assert_layer(self.name, kind, kernels, self.decode(kind, out), ref, absc,
                     emulate(op, st["x"], st["w"], st["b"], "act_residual_dropped"))

    def mt2(self, kind):
        """GC_CONV_MT2=1 sends this launch to k_me_conv with two M tiles per CTA (conv_layer.cu, launch)."""
        tiles = self.Ho * self.Wo // 128
        return kind == "planes" and self.taps == 9 and tiles % 2 == 0 and tiles * self.A >= 2 * 148


class DeconvCase:
    """ConvTranspose2d deblocks (kernel == stride == up) evaluated phase by phase as 1x1 GEMMs with a pixel-shuffle store
    (gc_conv_planes with up_dy = -1: all phases, fused into one launch where k_conv_tma applies), each level into its
    channel window of one shared output.  levels: (c_in, H, W, up, n_out)."""

    def __init__(self, name, A, levels, expect, kinds=("planes", "nchw"), launches=None):
        self.name, self.A, self.levels, self.expect, self.kinds = name, A, levels, expect, kinds
        self.launches = launches       # {kind: number of conv launches}
        self.Ho, self.Wo = levels[0][1] * levels[0][3], levels[0][2] * levels[0][3]
        assert all((h * up, w * up) == (self.Ho, self.Wo) for _, h, w, up, _ in levels)
        self.total = sum(lv[4] for lv in levels)
        self.n_tiles = A * self.Ho * self.Wo // 128
        self.stride, self.taps, self.many = 1, 1, False
        self.seed = sum(map(ord, name))

    def prepare(self, dev):
        from gencomm_b200 import ops
        lv = []
        for i, (c_in, h, w, up, n) in enumerate(self.levels):
            x = make_input(self.seed + 10 * i, self.A, c_in, h, w).to(dev)
            wt, b = make_weights(self.seed + 10 * i + 1, (c_in, n, up, up), c_in, n)
            wt, b = wt.to(dev), b.to(dev)
            phases = torch.cat([ops.conv_pack(wt[:, :, dy, dx].t().contiguous().view(n, c_in, 1, 1))
                                for dy in range(up) for dx in range(up)])
            lv.append({"x": x, "w": wt, "b": b, "planes": host_planes(x), "packed": phases})
        return {"levels": lv, "dev": dev}

    def launch(self, st, kind, check_windows=False):
        from gencomm_b200 import ops
        A, off = self.A, 0
        if kind == "planes":
            out = torch.full((2, A * self.Ho * self.Wo * self.total * 2), PLANE_FILL, dtype=torch.uint8, device=st["dev"])
        else:
            out = torch.full((A, self.total, self.Ho, self.Wo), float("nan"), device=st["dev"])
        for (c_in, h, w, up, n), L in zip(self.levels, st["levels"]):
            args = (L["planes"], A, c_in, h, w, L["packed"], L["b"], n, 1)
            if kind == "planes":
                ops.conv_planes(*args, out_planes=(out[0], out[1]), out_ch_total=self.total, out_ch_off=off, up=up, up_dy=-1)
            else:
                ops.conv_planes(*args, out_nchw=out, out_ch_off=off, up=up, up_dy=-1)
            off += n
            if check_windows:          # every phase covered every pixel of this window; later windows untouched
                if kind == "planes":
                    check_sentinel_planes(out, A, self.Ho, self.Wo, self.total, 0, off)
                else:
                    check_sentinel_nchw(out, 0, off)
        return out

    def decode(self, kind, out):
        if kind == "planes":
            return decode_planes(out, self.A, self.Ho, self.Wo, self.total, 0, self.total)
        return out.double()

    def split_matches(self, nchw, planes):
        assert_split_matches(nchw, planes, self.A, self.Ho, self.Wo, self.total, 0, self.total, self.name)

    def check(self, st, kind, out, kernels):
        out = self.launch(st, kind, check_windows=True)
        got, off = self.decode(kind, out), 0
        for (c_in, h, w, up, n), L in zip(self.levels, st["levels"]):
            op = conv_op("deconv", up)
            ref, absc = reference(op, L["x"], L["w"], L["b"])
            assert_layer(f"{self.name}@{off}", kind, kernels, got[:, off:off + n], ref, absc,
                         emulate(op, L["x"], L["w"], L["b"], "act_residual_dropped", in_dim=0))
            off += n

    def mt2(self, kind):
        return False


class HeadsCase:
    """gc_det_heads: one 1x1 GEMM (bias, no activation) for the concatenated cls / reg / dir heads over NCHW fp32 input."""

    def __init__(self, name, B, C, H, W, n_out, expect, many=False):
        self.name, self.A, self.C, self.H, self.W, self.n_out = name, B, C, H, W, n_out
        self.expect, self.kinds, self.many = expect, ("nchw",), many
        self.n_tiles = B * H * W // 128
        self.stride, self.taps = 1, 1
        self.seed = sum(map(ord, name))

    def prepare(self, dev):
        from gencomm_b200 import _lib, ops
        x = make_input(self.seed, self.A, self.C, self.H, self.W).to(dev)
        w, b = make_weights(self.seed + 1, (self.n_out, self.C, 1, 1), self.C, self.n_out)
        w, b = w.to(dev), b.to(dev)
        packed, bias, _ = ops.det_heads_pack([w], [b])
        lib = _lib.load()
        ws = torch.empty(lib.gc_det_heads_workspace_bytes(self.A, self.C, self.H, self.W), dtype=torch.uint8, device=dev)
        return {"x": x, "w": w, "b": b, "packed": packed, "bias": bias, "ws": ws}

    def launch(self, st, kind):
        from gencomm_b200 import _lib, ops
        lib = _lib.load()
        out = torch.full((self.A, self.n_out, self.H, self.W), float("nan"), device=st["x"].device)
        _lib.check(lib.gc_det_heads(ops._ptr(st["x"]), self.A, self.C, self.H, self.W, self.n_out, ops._ptr(st["packed"]),
                                    ops._ptr(st["bias"]), ops._ptr(st["ws"]), ops._ptr(out), ops._stream()), "gc_det_heads")
        return out

    def decode(self, kind, out):
        return out.double()

    def check(self, st, kind, out, kernels):
        check_sentinel_nchw(out, 0, self.n_out)
        op = conv_op("conv1")
        ref, absc = reference(op, st["x"], st["w"], st["b"], relu=False)
        assert_layer(self.name, kind, kernels, out.double(), ref, absc,
                     emulate(op, st["x"], st["w"], st["b"], "act_residual_dropped", relu=False))

    def mt2(self, kind):
        return False


def _tma(nout, taps, epi, mc, stg):
    return f"k_conv_tma<{nout},{taps},{epi},{mc},{stg}>"


def _me(nout, taps, epi, mt=1):
    return f"k_me_conv<{nout},0,32,{taps},{epi},{mt}>"


MATRIX = [
    # 1-2: the benched level-1 layers (64 ch): strided input through the TMA element strides, stride-1 body
    ConvCase("s2_64_256x512", 2, 64, 256, 512, 64, stride=2, many=True,
             expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("s1_64_128x256", 2, 64, 128, 256, 64, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    # 3-6: CTA pairs sharing every weight stage by multicast, three or more tiles per CTA
    ConvCase("s2_64to128_A8", 8, 64, 128, 256, 128, stride=2, many=True,
             expect={"planes": [_tma(128, 9, 5, 1, 1)], "nchw": [_tma(128, 9, 3, 1, 0)]}),
    ConvCase("s1_128_A8", 8, 128, 64, 128, 128, many=True,
             expect={"planes": [_tma(128, 9, 5, 1, 1)], "nchw": [_tma(128, 9, 3, 1, 0)]}),
    ConvCase("s2_128to256_A32", 32, 128, 64, 128, 256, stride=2, many=True,
             expect={"planes": [_tma(256, 9, 5, 1, 0)], "nchw": [_tma(256, 9, 3, 1, 0)]}),
    ConvCase("s1_256_A32_win128of512", 32, 256, 32, 64, 256, total=512, off=128, many=True,
             expect={"planes": [_tma(256, 9, 5, 1, 0)], "nchw": [_tma(256, 9, 3, 1, 0)]}),
    # 7: NOUT 256 without the pairs: an odd tile count, and fewer than 4 tiles
    ConvCase("s1_256_6x64_A5", 5, 256, 6, 64, 256, expect={"planes": [_tma(256, 9, 5, 0, 0)], "nchw": [_tma(256, 9, 3, 0, 0)]}),
    ConvCase("s1_256_2x128_A1", 1, 256, 2, 128, 256, expect={"planes": [_tma(256, 9, 5, 0, 0)], "nchw": [_tma(256, 9, 3, 0, 0)]}),
    # 8: the m1 backbone's three deblocks (up 1, 2, 4) into one 384-channel output
    DeconvCase("deblocks_384", 2, [(64, 64, 128, 1, 128), (128, 32, 64, 2, 128), (256, 16, 32, 4, 128)],
               expect={"planes": [_tma(128, 1, 5, 0, 1)], "nchw": [_tma(128, 1, 3, 0, 0)]}, launches={"planes": 3, "nchw": 3}),
    # 9: output widths below the kernel's N: the generic epilogue over zero-padded weights
    ConvCase("nout24", 4, 64, 32, 64, 24, expect={"nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("nout48", 4, 64, 32, 64, 48, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("nout80", 4, 64, 32, 64, 80, expect={"planes": [_tma(128, 9, 5, 1, 1)], "nchw": [_tma(128, 9, 3, 1, 0)]}),
    ConvCase("nout200", 4, 64, 32, 64, 200, expect={"nchw": [_tma(256, 9, 3, 1, 0)]}),
    ConvCase("nout240", 4, 64, 32, 64, 240, expect={"planes": [_tma(256, 9, 5, 1, 0)], "nchw": [_tma(256, 9, 3, 1, 0)]}),
    # 10: one and three 32-channel chunks per tap; 1x1 with a single stage per tile, ~7 tiles per CTA
    ConvCase("cin32_3x3", 2, 32, 64, 128, 64, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("cin96_3x3", 4, 96, 32, 64, 128, expect={"planes": [_tma(128, 9, 5, 1, 1)], "nchw": [_tma(128, 9, 3, 1, 0)]}),
    ConvCase("cin32_1x1_A4", 4, 32, 128, 256, 64, taps=1, many=True,
             expect={"planes": [_tma(64, 1, 5, 0, 1)], "nchw": [_tma(64, 1, 3, 0, 0)]}),
    ConvCase("cin96_1x1", 4, 96, 32, 64, 128, taps=1, expect={"planes": [_tma(128, 1, 5, 1, 1)], "nchw": [_tma(128, 1, 3, 1, 0)]}),
    # 11: narrow boxes (BW 32 x BH 4, BW 8 x BH 16), stride 1 and 2
    ConvCase("w32_s1", 3, 64, 16, 32, 64, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("w8_s1", 3, 64, 32, 8, 64, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("w32_s2", 3, 64, 32, 64, 64, stride=2, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("w8_s2", 3, 64, 64, 16, 64, stride=2, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    # 12: stride 2 over odd input sizes: the last tap of the last output column / row lies past the input
    ConvCase("odd_s2_65x255", 2, 64, 65, 255, 64, stride=2, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    ConvCase("odd_s2_15x63", 2, 64, 15, 63, 64, stride=2, expect={"planes": [_tma(64, 9, 5, 0, 1)], "nchw": [_tma(64, 9, 3, 0, 0)]}),
    # 13: widths TMA cannot tile (not a power of two, not a multiple of 128): k_me_conv, stride 1 and 2
    ConvCase("me_8x48_s1", 2, 64, 8, 48, 64, expect={"planes": [_me(64, 9, 5)], "nchw": [_me(64, 9, 3)]}),
    ConvCase("me_16x200_s1", 1, 64, 16, 200, 128, expect={"planes": [_me(128, 9, 5)], "nchw": [_me(128, 9, 3)]}),
    ConvCase("me_s2_16x96", 2, 64, 16, 96, 64, stride=2, expect={"planes": [_me(64, 9, 5)], "nchw": [_me(64, 9, 3)]}),
    ConvCase("me_s2_odd_15x95", 2, 64, 15, 95, 64, stride=2, expect={"planes": [_me(64, 9, 5)], "nchw": [_me(64, 9, 3)]}),
    ConvCase("me_s2_32x400", 1, 64, 32, 400, 64, stride=2, expect={"planes": [_me(64, 9, 5)], "nchw": [_me(64, 9, 3)]}),
    DeconvCase("deblock_me_w48", 2, [(128, 8, 48, 2, 64)], expect={"planes": [_me(64, 1, 5)], "nchw": [_me(64, 1, 3)]},
               launches={"planes": 4, "nchw": 4}),
    # 14: all phases requested with n_out < 64 on a TMA-eligible shape: one launch per phase
    DeconvCase("deblock_n48_loop", 2, [(64, 32, 64, 2, 48)], expect={"planes": [_tma(64, 1, 5, 0, 1)], "nchw": [_tma(64, 1, 3, 0, 0)]},
               launches={"planes": 4, "nchw": 4}),
    # 17: the V2X-Real heads (C = 256)
    HeadsCase("heads_C256_B8", 8, 256, 64, 128, 20, expect={"nchw": ["k_me_to_nhwc", _tma(32, 1, 0, 0, 0)]}, many=True),
]
CONV_KERNELS = ("k_conv_tma", "k_me_conv", "k_conv_rows")


def _conv_launches(kernels):
    return [k for k in kernels if k.startswith(CONV_KERNELS)]


@pytest.mark.parametrize("case", MATRIX, ids=lambda c: c.name)
def test_layer_matches_fp64(case):
    if case.many:
        sms = sm_count()
        assert case.n_tiles >= 3 * sms and case.n_tiles % sms, (case.name, case.n_tiles, sms)
    st = case.prepare(DEV)
    outs = {}
    for kind in case.kinds:
        _, kernels = launched(lambda: case.launch(st, kind))
        for k in case.expect.get(kind, []):
            assert any(n == k or n.startswith(k + "<") for n in kernels), f"{case.name}/{kind}: expected {k}, ran {kernels}"
        if getattr(case, "launches", None):
            assert len(_conv_launches(kernels)) == case.launches[kind], (case.name, kind, kernels)
        out = case.launch(st, kind)
        torch.cuda.synchronize()
        case.check(st, kind, out, _conv_launches(kernels) or kernels)
        outs[kind] = out
    if len(outs) == 2:
        case.split_matches(outs["nchw"], outs["planes"])


ROWS = [ConvCase("rows_64_128x256", 2, 64, 128, 256, 64, total=128, off=64, expect={"planes": ["k_conv_rows"], "nchw": ["k_conv_rows"]}),
        ConvCase("rows_128_64x128", 2, 128, 64, 128, 128, total=256, off=128, expect={"planes": ["k_conv_rows"], "nchw": ["k_conv_rows"]})]


@pytest.mark.parametrize("case", ROWS, ids=lambda c: c.name)
def test_conv_rows_matches_fp64(case, monkeypatch):
    """GC_CONV_ROWS=1 (read per call): the row-staged kernel accumulates chunk-major with the taps inside, k_conv_tma
    tap-major, so the two agree to the fp64 tolerance, not bit for bit."""
    monkeypatch.setenv("GC_CONV_ROWS", "1")
    test_layer_matches_fp64(case)


@pytest.mark.parametrize("A,C,H,W", [(3, 128, 7, 13), (2, 64, 32, 64), (1, 256, 1, 3)])
def test_to_planes_matches_host_split(A, C, H, W):
    from gencomm_b200 import ops
    x = make_input(A + C + H, A, C, H, W).to(DEV)
    (xh, xl), kernels = launched(lambda: ops.to_planes(x))
    assert kernels == ["k_me_to_nhwc"], kernels
    rh, rl = host_planes(x)
    assert torch.equal(xh, rh) and torch.equal(xl, rl)


def test_conv_planes_refusals():
    from gencomm_b200 import ops
    A, c, H, W = 1, 64, 8, 32
    x = make_input(3, A, c, H, W).to(DEV)
    planes = host_planes(x)
    w, b = make_weights(4, (64, c, 3, 3), 9 * c, 64)
    packed, b = ops.conv_pack(w.to(DEV)), b.to(DEV)
    out = torch.full((A, 64, H, W), float("nan"), device=DEV)
    with pytest.raises(RuntimeError, match="n_out % 8 == 0"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 20, 9, out_nchw=out)
    with pytest.raises(RuntimeError, match="plane outputs need n_out % 16 == 0"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 24, 9)
    with pytest.raises(RuntimeError, match="bad stride"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 64, 9, stride=3, out_nchw=out)
    with pytest.raises(RuntimeError, match="taps in"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 64, 4, out_nchw=out)
    with pytest.raises(RuntimeError, match="multiple of 128"):
        ops.conv_planes(planes, A, c, H, W - 2, packed, b, 64, 9, out_nchw=out)
    with pytest.raises(RuntimeError, match="bad output channel window"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 64, 9, out_nchw=out, out_ch_off=8)
    with pytest.raises(RuntimeError, match="up-sampling phase"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 64, 1, out_nchw=out, up=2, up_dy=2)
    with pytest.raises(RuntimeError, match="up-sampling phase"):
        ops.conv_planes(planes, A, c, H, W, packed, b, 64, 9, out_nchw=out, up=2, up_dy=-1)
    torch.cuda.synchronize()
    assert bool((out.view(torch.int32) == NAN_BITS).all()), "a refused call wrote its output"
    _, kernels = launched(lambda: ops.conv_planes(planes, 0, c, H, W, packed, b, 64, 9, out_nchw=out))
    assert kernels == [], kernels
    assert bool((out.view(torch.int32) == NAN_BITS).all())


# ------------------------------------------------------------------------------------------------
# the once-per-process switches, in child processes
# ------------------------------------------------------------------------------------------------
SWITCHES = {"tma0": {"GC_CONV_TMA": "0"}, "tma1": {"GC_CONV_TMA": "1"}, "mc0": {"GC_CONV_MC": "0"}, "mt2": {"GC_CONV_MT2": "1"}}


def run_matrix(dev):
    """{case/kind: (raw output on the CPU, kernels)} of every MATRIX launch on this process's path."""
    res = {}
    for case in MATRIX:
        st = case.prepare(dev)
        for kind in case.kinds:
            out, kernels = launched(lambda: case.launch(st, kind))
            res[f"{case.name}/{kind}"] = (out.cpu(), kernels)
    return res


@pytest.fixture(scope="module")
def default_outputs(tmp_path_factory):
    d = tmp_path_factory.mktemp("conv_switches")
    torch.save({k: v[0] for k, v in run_matrix(DEV).items()}, str(d / "default.pt"))
    return d


def _child_main(out_dir, tag):
    default = torch.load(os.path.join(out_dir, "default.pt"))
    report = {}
    for case in MATRIX:
        st = case.prepare(DEV)
        for kind in case.kinds:
            key = f"{case.name}/{kind}"
            out, kernels = launched(lambda: case.launch(st, kind))
            ref = default[key].to(DEV)
            same = torch.equal(out.view(torch.uint8), ref.view(torch.uint8))      # bit for bit, NaN sentinels included
            dmax = 0.0 if same else float((case.decode(kind, out) - case.decode(kind, ref)).abs().nan_to_num(float("inf")).max())
            report[key] = {"identical": same, "max_abs": dmax, "kernels": kernels}
    with open(os.path.join(out_dir, f"{tag}.json"), "w") as f:
        json.dump(report, f)


def _uses(kernels, prefix):
    return any(k.startswith(prefix) for k in kernels)


@pytest.mark.parametrize("tag", list(SWITCHES))
def test_switch_reproduces_default_bit_for_bit(tag, default_outputs):
    """GC_CONV_TMA=0 (k_me_conv everywhere), =1 (k_conv_tma at stride 1 only), GC_CONV_MC=0 (no CTA pairs), GC_CONV_MT2=1
    (two M tiles per CTA for 3x3 plane layers): same packed weights, same tap-major stage order, same epilogues -- the
    outputs of every case equal the default path's bit for bit."""
    env = dict(os.environ, **SWITCHES[tag])
    flags = [f for f, on in (("-I", sys.flags.isolated), ("-s", sys.flags.no_user_site), ("-E", sys.flags.ignore_environment)) if on]
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), str(default_outputs), tag], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    with open(default_outputs / f"{tag}.json") as f:
        report = json.load(f)
    cases = {c.name: c for c in MATRIX}
    for key, rec in report.items():
        name, kind = key.split("/")
        case, conv = cases[name], _conv_launches(rec["kernels"])
        assert conv, (key, rec["kernels"])
        if tag == "tma0":
            assert not _uses(conv, "k_conv_tma"), (key, conv)
        elif tag == "tma1":
            assert _uses(conv, "k_conv_tma") != (case.stride == 2 or not _uses(case.expect[kind], "k_conv_tma")), (key, conv)
        elif tag == "mc0":
            assert all(template_args(k)[3] == "0" for k in conv if k.startswith("k_conv_tma")), (key, conv)
        elif tag == "mt2":
            n = getattr(case, "n_out", 0)
            nout = 64 if n <= 64 else 128 if n <= 128 else 256
            assert (_me(nout, 9, 5, 2) in conv) == case.mt2(kind), (key, conv)
    bad = {k: v["max_abs"] for k, v in report.items() if not v["identical"]}
    assert not bad, f"{tag}: outputs differ from the default path (case: max |d|): {bad}"
    assert len(report) == sum(len(c.kinds) for c in MATRIX)


if __name__ == "__main__":
    _child_main(sys.argv[1], sys.argv[2])
