"""Every layer of the DiffusionUNet denoiser on its own, the cluster-resident middle included, against a float64 reference.

gc_unet_trace runs one evaluation exactly like gc_unet_forward and also writes hs0 (the conv_in output) and the output of each
of the 26 middle layers.  Each layer is then recomputed in float64 from ITS OWN inputs taken from that trace, so that errors do
not accumulate from layer to layer, with the fp32 record of step t of the host blob (pack_unet: weights, bias + that step's
timestep-embedding projection, GroupNorm affine, nin_shortcut):

  * element-wise  |got - ref| <= KAPPA[arith] * E,   E = conv(|a|, |w|) + conv(|xhat|, |w|) / 4 + |b| + |residual terms|,
    where a is the conv operand (swish of the GroupNorm output xhat, or the raw input) -- the xhat term covers the absolute
    error of the cluster kernel's fp16 tanh (about |xhat| 2^-12 in a) and of the GroupNorm statistics, which rstd (up to 1e3
    at eps 1e-6) amplifies;
  * aggregate     ||got - ref||_2 / ||ref||_2 <= RHO[arith], per agent;
  * sensitivity   fp64 emulations of a broken layer exceed both bounds on every case: (a) the halo rows across the row-band
    boundaries read as zero and (c) on conv1 layers the bias record of the neighbouring timestep by SENS x, (b) GroupNorm
    statistics of the band only by SENS_BANDS x;
  * sentinels     trace and pred start as NaN: every element is written and finite;
  * identity      pred of gc_unet_trace == pred of gc_unet_forward bit for bit (ties the dump instantiation of the cluster
    kernel to the production one), a repeated call is bit-identical, PREC_TC_MATERIALIZE changes nothing;
  * kernels       torch.profiler shows which conv_in / middle / conv_out kernels ran (and which did not).

One KAPPA / RHO per arithmetic (how each kernel rounds, from the code):
  "fp32"  k_conv_in / k_conv_c8 / k_conv_out and the cluster's downsample: fp32 FMAs;
  "tf32"  k_conv_c8_tc and the cluster's upsample: fp32 operands read by kind::tf32 MMAs (the low 13 mantissa bits are not used;
          the weights are not pre-rounded), fp32 accumulation in TMEM;
  "cl"    the cluster's GroupNorm layers: as "tf32", with swish = h + h tanh(h), h = xhat / 2, tanh.approx.f16x2 on
          fp16-rounded h (absolute error ~2^-11), and GroupNorm band sums combined in fp32;
  "bf16"  k_conv_in_tc / k_conv_in_tc2 / k_conv_out_tc: round-to-nearest bf16 operands, fp32 accumulation.
The constants and helpers here are shared with test_denoiser_tolerance_cpu.py, which checks the tolerance model on the CPU.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

# Per-layer bounds per arithmetic (DESIGN.md 5), set from B200 measurements (NVIDIA B200, 1000 W limit) of this file's cases,
# max |d| / E and max per-agent rms:
#   fp32  1.9e-4 / 2.7e-4: the unfused kernels' per-tile fp32 sums of squares on the DC-offset inputs (layers 0, 3, 24; an
#         rstd error of ~1e-4), <= 2e-6 everywhere else;
#   tf32  8.3e-4 / 1.2e-3 (the upsample, layer 19);   cl  6.3e-4 / 1.1e-3;   bf16  2.4e-3 / 2.5e-3 (conv_out, C = 8 conv_in).
# The CPU emulations (test_denoiser_tolerance_cpu.py) reach fp32 3e-7, tf32 7e-4 / 8e-4, cl 3e-4 / 1.1e-3, bf16 1.7e-3 / 2.3e-3.
KAPPA = {"fp32": 1e-3, "tf32": 4e-3, "cl": 4e-3, "bf16": 1.5e-2}
RHO = {"fp32": 1.5e-3, "tf32": 5e-3, "cl": 6e-3, "bf16": 1.5e-2}
SENS = 5.0          # a broken emulation must exceed both bounds by this factor; a correct emulation must stay SENS x below
# (b), GroupNorm statistics of the CTA's own row band only, changes a 64 x 128 layer by a few per cent of E: it is held to 2 x.
# Measured minimum on the cluster cases: 2.6 x (one agent, layer 13); (a) >= 7.9 x, (c) >= 9.6 x.
SENS_BANDS = 2.0
DC_RATIO = 30.0     # group mean / group std of the offset inputs (conv_in output of agent 0, the output of DC_LAYER)
DC_LAYER = 2        # down.0.block.1 conv1: its output is the GroupNorm input of layer 3
TEMB_SCALE = 10.0   # temb_proj weights x this: the step's bias differs enough from the neighbouring step's for check (c)

pytestmark = pytest.mark.gpu
DEV = "cuda"

# ------------------------------------------------------------------------------------------------
# layer table: mirrors c_layers of csrc/denoiser_cluster.cu and the launch order of unet_eval in csrc/denoiser.cu, in trace
# tensor indices (0 = hs0, 1 + l = output of layer l).  (kind, in_a, in_b, res, res_a, res_b, conv1)
# ------------------------------------------------------------------------------------------------
LAYERS = [
    ("conv", 0, None, None, None, None, True),     # 0  down.0.block.0 conv1
    ("conv", 1, None, "ident", 0, None, False),    # 1                 conv2 + x       -> hs1 = T2
    ("conv", 2, None, None, None, None, True),     # 2  down.0.block.1 conv1
    ("conv", 3, None, "ident", 2, None, False),    # 3                 conv2 + x       -> hs2 = T4
    ("down", 4, None, None, None, None, False),    # 4  down.0.downsample              -> hs3 = T5
    ("conv", 5, None, None, None, None, True),     # 5  down.1.block.0 conv1
    ("conv", 6, None, "ident", 5, None, False),    # 6                                 -> hs4 = T7
    ("conv", 7, None, None, None, None, True),     # 7  down.1.block.1 conv1
    ("conv", 8, None, "ident", 7, None, False),    # 8                                 -> hs5 = T9
    ("conv", 9, None, None, None, None, True),     # 9  mid.block_1 conv1
    ("conv", 10, None, "ident", 9, None, False),   # 10
    ("conv", 11, None, None, None, None, True),    # 11 mid.block_2 conv1
    ("conv", 12, None, "ident", 11, None, False),  # 12
    ("conv", 13, 9, None, None, None, True),       # 13 up.1.block.0 conv1 on cat(h, hs5)
    ("conv", 14, None, "nin", 13, 9, False),       # 14              conv2 + nin(cat)
    ("conv", 15, 7, None, None, None, True),       # 15 up.1.block.1 (hs4)
    ("conv", 16, None, "nin", 15, 7, False),       # 16
    ("conv", 17, 5, None, None, None, True),       # 17 up.1.block.2 (hs3)
    ("conv", 18, None, "nin", 17, 5, False),       # 18
    ("up", 19, None, None, None, None, False),     # 19 up.1.upsample (nearest x2 + 3x3)
    ("conv", 20, 4, None, None, None, True),       # 20 up.0.block.0 (hs2)
    ("conv", 21, None, "nin", 20, 4, False),       # 21
    ("conv", 22, 2, None, None, None, True),       # 22 up.0.block.1 (hs1)
    ("conv", 23, None, "nin", 22, 2, False),       # 23
    ("conv", 24, 0, None, None, None, True),       # 24 up.0.block.2 (hs0)
    ("conv", 25, None, "nin", 24, 0, False),       # 25                                -> input of norm_out = T26
]
N_LAYERS = len(LAYERS)
C8_FLOATS = 1328                                    # sizeof(C8Params) / 4
PREC_CLUSTER = 16


def is_half(k):
    """Trace tensor k is half resolution (layers 4 .. 18)."""
    return 5 <= k <= 19


# ------------------------------------------------------------------------------------------------
# host helpers (device-agnostic; test_denoiser_tolerance_cpu.py runs them on the CPU)
# ------------------------------------------------------------------------------------------------
def cfg(C):
    return {"model": {"embed_dim": C + 2, "in_channels": C, "out_ch": C, "ch": 8, "ch_mult": [1, 1],
                      "num_res_blocks": 2, "attn_resolutions": [16], "dropout": 0.0, "resamp_with_conv": True},
            "diffusion": {"beta_schedule": "linear", "beta_start": 0.0005, "beta_end": 0.02,
                          "num_diffusion_timesteps": 3}}


def random_sd(C, seed):
    """state_dict (without the 'denoiser.' prefix) of a random DiffusionUNet: default init, GroupNorm affine and biases
    perturbed, temb_proj x TEMB_SCALE, and DC_LAYER's bias raised so that its output has a group mean ~DC_RATIO x its std."""
    import gencomm_b200 as G
    torch.manual_seed(seed)
    m = G.GenComm(cfg(C)).denoiser
    sd = {k: v.detach().clone().float() for k, v in m.state_dict().items()}
    for k, v in sd.items():
        if "norm" in k:
            v.add_(0.2 * torch.randn_like(v))
        elif k.endswith(".bias"):
            v.add_(0.05 * torch.randn_like(v))
        if ".temb_proj." in k:
            v.mul_(TEMB_SCALE)
    # the conv output over normalised, swish-activated inputs has std ~0.35 for this init (fan-in 72)
    assert _layer_names()[DC_LAYER] == ("down.0.block.1", "conv1")
    sd["down.0.block.1.conv1.bias"] += DC_RATIO * 0.35
    return sd


def make_inputs(seed, A, C, H, W):
    """(cond [A,2,H,W], x [A,C,H,W]) fp32: agent a scaled by its own factor (1e-2 .. 1e2), border rows / columns x4, ~30 %
    exact zeros; agent 1 is all zeros; agent 0 (scale 1e-2) gets the conv_in bias offset (conv_in_dc_bias)."""
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(A, C + 2, H, W, generator=g)
    v[:, :, 0] *= 4.0
    v[:, :, -1] *= 4.0
    v[:, :, :, 0] *= 4.0
    v[:, :, :, -1] *= 4.0
    v[torch.rand(A, C + 2, H, W, generator=g) < 0.3] = 0.0
    scales = torch.logspace(2, -2, max(A - 2, 1)).tolist()
    s = [1e-2] + ([0.0] + scales if A > 1 else [])
    v *= torch.tensor(s[:A]).view(A, 1, 1, 1)
    return v[:, :2].contiguous(), v[:, 2:].contiguous()


def conv_in_dc_bias(sd, cond, x):
    """conv_in bias that puts agent 0's conv_in output at a group mean of DC_RATIO x its group std."""
    y = F.conv2d(torch.cat([cond[:1], x[:1]], 1).double(), sd["conv_in.weight"].double().to(x.device), padding=1)
    std = y.view(4, -1).std(dim=1)                         # 4 groups of 2 channels
    return (DC_RATIO * std).repeat_interleave(2).float().cpu()


def records(host, t, T=None):
    """The 26 fp32 C8Params records of step t of a pack_unet host blob as float64 tensors: w [8, cin, 3, 3], bias [8], gamma /
    beta [cin], nin_w [8, 16, 1, 1], nin_b [8] (layout: csrc/denoiser_tc.cuh)."""
    recs = torch.from_numpy(np.asarray(host[(t * N_LAYERS) * C8_FLOATS:(t + 1) * N_LAYERS * C8_FLOATS])).double()
    out = []
    for l, L in enumerate(LAYERS):
        r = recs[l * C8_FLOATS:(l + 1) * C8_FLOATS]
        cin = 16 if L[2] is not None else 8
        w = r[:1152].view(3, 3, 16, 8)[:, :, :cin, :].permute(3, 2, 0, 1).contiguous()
        out.append({"w": w, "bias": r[1152:1160].clone(), "gamma": r[1160:1160 + cin].clone(),
                    "beta": r[1176:1176 + cin].clone(), "nin_w": r[1192:1320].view(16, 8).t().reshape(8, 16, 1, 1).clone(),
                    "nin_b": r[1320:1328].clone()})
    return out


def records_from_sd(sd, t, temb_fn):
    """The same records computed from a float64 state_dict (the CPU chain check), temb_fn(t) = the [1, 32] embedding MLP
    output before swish."""
    names = _layer_names()
    act = _swish(temb_fn(t))
    out = []
    for l, (name, part) in enumerate(names):
        L = LAYERS[l]
        cin = 16 if L[2] is not None else 8
        if part is None:
            rec = {"w": sd[name + ".weight"], "bias": sd[name + ".bias"]}
        else:
            rec = {"w": sd[f"{name}.{part}.weight"], "bias": sd[f"{name}.{part}.bias"].clone()}
            norm = "norm1" if part == "conv1" else "norm2"
            rec["gamma"], rec["beta"] = sd[f"{name}.{norm}.weight"], sd[f"{name}.{norm}.bias"]
            if part == "conv1":
                rec["bias"] = rec["bias"] + F.linear(act, sd[name + ".temb_proj.weight"], sd[name + ".temb_proj.bias"])[0]
            if L[3] == "nin":
                rec["nin_w"], rec["nin_b"] = sd[name + ".nin_shortcut.weight"], sd[name + ".nin_shortcut.bias"]
        assert rec["w"].shape[1] == (cin if L[0] == "conv" else 8)
        out.append(rec)
    return out


def _layer_names():
    names = []
    for lvl in range(2):
        for blk in range(2):
            names += [(f"down.{lvl}.block.{blk}", "conv1"), (f"down.{lvl}.block.{blk}", "conv2")]
        if lvl == 0:
            names.append(("down.0.downsample.conv", None))
    for b in ("mid.block_1", "mid.block_2"):
        names += [(b, "conv1"), (b, "conv2")]
    for lvl in (1, 0):
        for blk in range(3):
            names += [(f"up.{lvl}.block.{blk}", "conv1"), (f"up.{lvl}.block.{blk}", "conv2")]
        if lvl == 1:
            names.append(("up.1.upsample.conv", None))
    return names


def _swish(v):
    return v * torch.sigmoid(v)


def band_rows(h):
    """Rows per band of the cluster kernel's 8 row bands (at least one row)."""
    return max(h // 8, 1)


def group_norm(x, gamma, beta, bands=False):
    """GroupNorm(4, eps 1e-6) of x [A, c, h, w] in the dtype of x; bands: statistics of each row band only (broken (b))."""
    A, c, h, w = x.shape
    if not bands:
        xg = x.reshape(A, 4, -1)
        mean, var = xg.mean(-1, keepdim=True), xg.var(-1, unbiased=False, keepdim=True)
        xh = ((xg - mean) / torch.sqrt(var + 1e-6)).view(A, c, h, w)
    else:
        r = band_rows(h)
        parts = [group_norm(x[:, :, y:y + r], torch.ones_like(gamma), torch.zeros_like(beta)) for y in range(0, h, r)]
        xh = torch.cat(parts, 2)
    return xh * gamma.view(1, -1, 1, 1) + beta.view(1, -1, 1, 1)


def _conv3(a, w, kind, halo_zero=False):
    if kind == "up":
        a = F.interpolate(a, scale_factor=2.0, mode="nearest")
    if kind == "down":
        return F.conv2d(F.pad(a, (0, 1, 0, 1)), w, stride=2)
    if not halo_zero:
        return F.conv2d(a, w, padding=1)
    r = band_rows(a.shape[2])
    return torch.cat([F.conv2d(F.pad(a[:, :, y:y + r], (1, 1, 1, 1)), w) for y in range(0, a.shape[2], r)], 2)


def layer_forward(l, ins, rec, dt=torch.float64, mode="exact", rec_alt=None, act=_swish, rnd=None):
    """Layer l of LAYERS on its inputs ins = (in_a, in_b or None, res_a or None, res_b or None) NCHW -> (out, E) in dtype dt.
    mode: "exact"; "halo" (a), "bands" (b), "bias" (c, rec_alt = the neighbouring step's record).  Emulations: act(xhat) is the
    activation, rnd rounds both operands of the 3x3 convolution."""
    kind, _, _, res, _, _, conv1 = LAYERS[l]
    ia, ib, ra, rb = (None if v is None else v.to(dt) for v in ins)
    x = ia if ib is None else torch.cat([ia, ib], 1)
    w, b = rec["w"].to(dt).to(x.device), rec["bias"].to(dt).to(x.device)
    if mode == "bias" and conv1:
        b = rec_alt["bias"].to(dt).to(x.device)
    xh = None
    if kind == "conv":
        # the GroupNorm coefficients in float64 (the unfused kernels combine their partial sums in double)
        xh = group_norm(x.double(), rec["gamma"].double().to(x.device), rec["beta"].double().to(x.device),
                        bands=(mode == "bands")).to(dt)
        a = act(xh).to(dt)
    else:
        a = x
    y = _conv3(rnd(a) if rnd else a, rnd(w) if rnd else w, kind, halo_zero=(mode == "halo")) + b.view(1, -1, 1, 1)
    E = _conv3(a.abs(), w.abs(), kind) + b.abs().view(1, -1, 1, 1)
    if xh is not None:   # the activation's absolute error: fp16 tanh of h = xhat / 2 errs by ~|xhat| 2^-12 in a
        E = E + 0.25 * _conv3(xh.abs(), w.abs(), kind)
    if res == "ident":
        y, E = y + ra, E + ra.abs()
    elif res == "nin":
        cat = torch.cat([ra, rb], 1)
        nw, nb = rec["nin_w"].to(dt).to(x.device), rec["nin_b"].to(dt).to(x.device)
        y = y + F.conv2d(cat, nw, nb)
        E = E + F.conv2d(cat.abs(), nw.abs(), nb.abs())
    return y, E


def layer_inputs(l, T):
    """(in_a, in_b, res_a, res_b) of layer l from a list T of NCHW tensors (trace order)."""
    _, ia, ib, _, ra, rb, _ = LAYERS[l]
    return tuple(None if k is None else T[k] for k in (ia, ib, ra, rb))


def conv_in_forward(cond, x, w, b, dt=torch.float64, rnd=None):
    inp = torch.cat([cond, x], 1).to(dt)
    w, b = w.to(dt).to(inp.device), b.to(dt).to(inp.device)
    y = F.conv2d(rnd(inp), rnd(w), b, padding=1) if rnd else F.conv2d(inp, w, b, padding=1)
    return y, F.conv2d(inp.abs(), w.abs(), b.abs(), padding=1)


def conv_out_forward(h, gamma, beta, w, b, dt=torch.float64, rnd=None):
    h = h.to(dt)
    xh = group_norm(h, gamma.to(dt).to(h.device), beta.to(dt).to(h.device))
    a = _swish(xh)
    w, b = w.to(dt).to(h.device), b.to(dt).to(h.device)
    return (F.conv2d(rnd(a), rnd(w), b, padding=1) if rnd else F.conv2d(a, w, b, padding=1),
            F.conv2d(a.abs(), w.abs(), b.abs(), padding=1) + 0.25 * F.conv2d(xh.abs(), w.abs(), padding=1))


def rel_errors(got, ref, E):
    """(max |got - ref| / E, max over agents of ||got - ref||_2 / ||ref||_2); where E is 0 the reference is exactly 0 and so
    must be the result.  The aggregate is per agent: the agents' scales span 1e4, and the identity residuals carry them."""
    d = (got.double() - ref).abs()
    elem = torch.where(E > 0, d / E.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    A = ref.shape[0]
    rms = d.reshape(A, -1).norm(dim=1) / ref.reshape(A, -1).norm(dim=1).clamp_min(1e-300)
    return float(elem.max()), float(rms.max())


def passes(errs, arith):
    return errs[0] <= KAPPA[arith] and errs[1] <= RHO[arith]


def nhwc_to_nchw(t):
    return t.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------
# which kernel runs where: mirrors unet_eval (csrc/denoiser.cu) and the eligibility rules of csrc/denoiser_tc.cu
# ------------------------------------------------------------------------------------------------
def conv_in_tc_ok(C, H, W):
    chunks = (C // 8 + 2) // 2
    return W % 128 == 0 and C % 8 == 0 and C >= 8 and 2 * 2 * 6 * 130 * 16 + chunks * 9 * 2 * 128 <= 200 * 1024


def conv_in_tc2_ok(C, H, W):
    chunks = (C // 8 + 2) // 2
    return W == 128 and H % 8 == 0 and C % 8 == 0 and C >= 8 and 2 * 41600 + chunks * 3 * 1024 <= 220 * 1024


def conv_out_tc_ok(C, H, W):
    return W % 128 == 0 and C % 64 == 0


def plan(prec, C, H, W, conv_in_v1=False):
    """(conv_in kernel, conv_out kernel, arithmetic of each middle layer, cluster?)."""
    cluster = bool(prec & PREC_CLUSTER) and prec & 3 == 3 and (H, W) == (64, 128) and conv_in_tc_ok(C, H, W) \
        and conv_out_tc_ok(C, H, W)
    if (cluster or prec & 1) and conv_in_tc2_ok(C, H, W) and not conv_in_v1:
        cin = "k_conv_in_tc2"
    elif (cluster or prec & 1) and conv_in_tc_ok(C, H, W):
        cin = "k_conv_in_tc"
    else:
        cin = "k_conv_in"
    cout = "k_conv_out_tc" if (cluster or prec & 2) and conv_out_tc_ok(C, H, W) else "k_conv_out"
    mids = []
    for l, L in enumerate(LAYERS):
        w = W // 2 if is_half(l + 1) else W
        if cluster:
            mids.append("fp32" if L[0] == "down" else ("tf32" if L[0] == "up" else "cl"))
        else:
            mids.append("tf32" if prec & 8 and L[0] != "down" and w % 128 == 0 else "fp32")
    return cin, cout, mids, cluster


# ------------------------------------------------------------------------------------------------
# GPU cases
# ------------------------------------------------------------------------------------------------
# (precision, C, H, W, A, t)
CASES = [
    (27, 64, 64, 128, 1, 0),      # cluster, one agent
    (27, 128, 64, 128, 4, 1),     # cluster, conv_out N = 128
    (27, 192, 64, 128, 20, 2),    # cluster, conv_out N = 64 x 3 splits, more agents than one round
    (27, 256, 64, 128, 61, 1),    # cluster, the bench's four rounds over the co-resident clusters, one agent in the last
    (11, 64, 64, 128, 3, 2),      # tc: tf32 middle at 64 x 128, conv_in_tc2, conv_out_tc
    (1, 64, 64, 128, 2, 0),       # bf16 conv_in only
    (2, 128, 64, 128, 2, 1),      # bf16 conv_out only
    (3, 64, 64, 128, 3, 2),       # bf16 conv_in + conv_out, fp32 middle
    (8, 64, 64, 128, 3, 0),       # tf32 middle only
    (11, 64, 8, 128, 3, 1),       # a single 8-row conv_in band
    (27, 64, 72, 128, 3, 2),      # conv_in_tc2 but not cluster-eligible: falls back to 'tc'
    (11, 64, 16, 256, 3, 0),      # conv_in v1, two 128-pixel tiles per row, tf32 half-resolution layers
    (8, 64, 16, 256, 2, 2),       # tf32 middle only at W = 256
    (11, 8, 16, 128, 3, 1),       # C = 8: conv_in K below one 16-channel chunk, conv_out falls back to fp32
    (11, 728, 8, 128, 2, 2),      # the largest C conv_in_tc2 accepts
    (11, 736, 8, 128, 2, 0),      # the next multiple of 8: conv_in v1
    (0, 32, 20, 50, 3, 1),        # fp32
    (0, 64, 8, 34, 3, 2),         # fp32, half resolution 4 x 17
    (11, 64, 8, 34, 3, 0),        # 'tc' on an ineligible shape: everything fp32
]
T_STEPS = 3


def case_id(c):
    return f"p{c[0]}_C{c[1]}_{c[2]}x{c[3]}_A{c[4]}_t{c[5]}"


_built = {}


def build_case(case):
    """(sd, host, w_dev, w_cluster, cond, x) of a case, on the GPU; cached per case."""
    if case in _built:
        return _built[case]
    from gencomm_b200.gencomm import pack_unet, pack_unet_cluster
    prec, C, H, W, A, t = case
    sd = random_sd(C, seed=C + H + W + A)
    cond, x = make_inputs(1000 + C + H + A, A, C, H, W)
    sd["conv_in.bias"] = conv_in_dc_bias(sd, cond.to(DEV), x.to(DEV))
    host, dev = pack_unet(sd, C, T_STEPS)
    cl = torch.from_numpy(pack_unet_cluster(host, T_STEPS)).to(DEV)
    _built.clear()
    _built[case] = (sd, host, dev.to(DEV), cl, cond.to(DEV), x.to(DEV))
    return _built[case]


def run_trace(case, precision=None):
    from gencomm_b200 import ops
    prec, C, H, W, A, t = case
    sd, host, dev, cl, cond, x = build_case(case)
    lib = __import__("gencomm_b200._lib", fromlist=["load"]).load()
    pred = torch.full_like(x, float("nan"))
    trace = torch.full((lib.gc_unet_trace_floats(A, H, W),), float("nan"), device=DEV)
    p = prec if precision is None else precision
    pred, tensors = ops.unet_trace(cond, x, t, host, dev, T_STEPS, precision=p, w_cluster=cl, pred=pred, trace=trace)
    torch.cuda.synchronize()
    return pred, trace, tensors


def check_layers(case, pred, tensors, conv_in_v1=False):
    """Every layer against its float64 reference; returns the per-arithmetic measurements and the sensitivity ratios."""
    prec, C, H, W, A, t = case
    sd, host, dev, cl, cond, x = build_case(case)
    cin_k, cout_k, mids, _ = plan(prec, C, H, W, conv_in_v1)
    Tn = [nhwc_to_nchw(v) for v in tensors]
    recs = records(host, t)
    recs_alt = records(host, t + 1 if t + 1 < T_STEPS else t - 1)
    worst, sens, bad = {}, {}, []

    def note(arith, what, errs):
        m = worst.setdefault(arith, [0.0, 0.0, ""])
        if errs[0] > m[0]:
            m[0], m[2] = errs[0], what
        m[1] = max(m[1], errs[1])
        if not passes(errs, arith):
            bad.append((what, arith, errs))

    ref, E = conv_in_forward(cond, x, sd["conv_in.weight"], sd["conv_in.bias"])
    note("bf16" if cin_k != "k_conv_in" else "fp32", "conv_in", rel_errors(Tn[0], ref, E))
    for l in range(N_LAYERS):
        ins = layer_inputs(l, Tn)
        ref, E = layer_forward(l, ins, recs[l])
        arith = mids[l]
        note(arith, f"layer {l}", rel_errors(Tn[l + 1], ref, E))
        # DC_LAYER's output is dominated by its large bias: no rms bound can see a broken halo or statistics there
        modes = ["halo"] if LAYERS[l][0] != "down" and l != DC_LAYER else []
        modes += ["bands"] if LAYERS[l][0] == "conv" and l != DC_LAYER else []
        modes += ["bias"] if LAYERS[l][6] and l != DC_LAYER else []
        for mode in modes:
            if mode == "halo" and band_rows(ref.shape[2]) >= ref.shape[2]:
                continue                                # a single band: no boundary
            got, _ = layer_forward(l, ins, recs[l], mode=mode, rec_alt=recs_alt[l])
            e = rel_errors(got, ref, E)
            r = min(e[0] / KAPPA[arith], e[1] / RHO[arith])
            if r < sens.get(mode, (math.inf,))[0]:
                sens[mode] = (r, l)
    ref, E = conv_out_forward(Tn[26], sd["norm_out.weight"], sd["norm_out.bias"], sd["conv_out.weight"], sd["conv_out.bias"])
    note("bf16" if cout_k == "k_conv_out_tc" else "fp32", "conv_out", rel_errors(pred, ref, E))
    return worst, sens, bad


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_every_layer_against_fp64(case):
    pred, trace, tensors = run_trace(case)
    assert torch.isfinite(trace).all(), "trace element not written or not finite"
    assert torch.isfinite(pred).all(), "pred element not written or not finite"
    worst, sens, bad = check_layers(case, pred, tensors)
    print(f"\n[layers] {case_id(case)} " + " ".join(f"{k}: max {v[0]:.2e} ({v[2]}) rms {v[1]:.2e}" for k, v in worst.items())
          + " | sensitivity " + " ".join(f"{k}: {v[0]:.1f}x (layer {v[1]})" for k, v in sens.items()))
    assert not bad, bad
    for mode, (r, l) in sens.items():
        assert r >= (SENS_BANDS if mode == "bands" else SENS), (mode, l, r)


def _kernels(fn):
    """Names of the GPU activities of fn.  The profiler can lose the first activities of its window (a run missed the
    Memcpy and k_conv_in that open every evaluation), so fn runs twice and the names of both runs count: "ran" then means
    ran in at least one run, "not ran" in neither."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as p:
        for _ in range(2):
            fn()
            torch.cuda.synchronize()
    return {e.name for e in p.events() if e.device_type.name == "CUDA"}


def _bare(names):
    """Kernel names without return type, namespace, template arguments and parameters."""
    return {n.removeprefix("void ").split("(")[0].split("<")[0].split("::")[-1] for n in names}


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_trace_identity_and_kernels(case):
    """pred of gc_unet_trace == pred of gc_unet_forward bit for bit; the trace is deterministic; the planned kernels ran."""
    from gencomm_b200 import ops
    prec, C, H, W, A, t = case
    sd, host, dev, cl, cond, x = build_case(case)
    cin_k, cout_k, mids, cluster = plan(prec, C, H, W)
    names = _kernels(lambda: run_trace(case))
    pred, trace, _ = run_trace(case)
    pred2, trace2, _ = run_trace(case)
    assert torch.equal(pred, pred2) and torch.equal(trace, trace2), "repeated gc_unet_trace differs"
    fwd_names = _kernels(lambda: ops.unet_forward(cond, x, t, host, dev, T_STEPS, precision=prec, w_cluster=cl))
    fwd = ops.unet_forward(cond, x, t, host, dev, T_STEPS, precision=prec, w_cluster=cl)
    assert torch.equal(pred, fwd), "gc_unet_trace pred differs from gc_unet_forward"
    bare, fwd_bare = _bare(names), _bare(fwd_names)
    for k in {"k_conv_in", "k_conv_in_tc", "k_conv_in_tc2", "k_conv_out", "k_conv_out_tc"}:
        assert (k in bare) == (k in (cin_k, cout_k)), ("gc_unet_trace", k, sorted(bare))
        assert (k in fwd_bare) == (k in (cin_k, cout_k)), ("gc_unet_forward", k, sorted(fwd_bare))
    if cluster:
        assert any("k_unet_middle_cluster<true>" in n for n in names), sorted(names)
        assert any("k_unet_middle_cluster<false>" in n for n in fwd_names), sorted(fwd_names)
        assert not any("k_unet_middle_cluster<false>" in n for n in names)
        assert "k_conv_c8" not in bare and "k_conv_c8_tc" not in bare
    else:
        assert "k_unet_middle_cluster" not in bare | fwd_bare
        assert "k_conv_c8" in bare                                    # the downsample at least
        assert ("k_conv_c8_tc" in bare) == ("tf32" in mids), sorted(bare)
    if prec & 3 == 3 and not cluster:
        mat = ops.unet_forward(cond, x, t, host, dev, T_STEPS, precision=prec | ops.PREC_TC_MATERIALIZE, w_cluster=cl)
        assert torch.equal(mat, fwd), "PREC_TC_MATERIALIZE changes the result"


@pytest.mark.parametrize("case", [CASES[1], CASES[10]], ids=case_id)
def test_conv_in_v1_switch(case, monkeypatch):
    """GC_CONV_IN_V1 (read per call) selects k_conv_in_tc instead of k_conv_in_tc2; the layers stay within their bounds."""
    monkeypatch.setenv("GC_CONV_IN_V1", "1")
    names = _kernels(lambda: run_trace(case))
    assert "k_conv_in_tc" in _bare(names) and "k_conv_in_tc2" not in _bare(names), sorted(names)
    pred, trace, tensors = run_trace(case)
    worst, _, bad = check_layers(case, pred, tensors, conv_in_v1=True)
    assert not bad, bad


def test_trace_refuses_null_trace():
    from gencomm_b200 import _lib
    lib = _lib.load()
    assert lib.gc_unet_trace(None, None, 1, 0, None, None, None, 8, 8, 8, 3, 0, None, None, None, None) != 0
    assert lib.gc_unet_trace_floats(2, 8, 16) == 2 * (12 * 8 * 16 * 8 + 15 * 4 * 8 * 8)
