"""The tolerance model of test_denoiser_layers_gpu.py, on the CPU.

A float64 emulation of each arithmetic the denoiser kernels use must pass the per-layer bounds KAPPA / RHO with a SENS x margin,
and every emulation of a broken layer must exceed both bounds by SENS x -- otherwise the GPU test could not tell a correct
kernel from a broken one.  The test's layer table, chained in float64 on exact inputs, must reproduce ref_ops.unet_forward.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_ops as R
from test_denoiser_layers_gpu import (DC_LAYER, KAPPA, LAYERS, N_LAYERS, RHO, SENS, SENS_BANDS, T_STEPS, conv_in_dc_bias,
                                      conv_in_forward,
                                      conv_out_forward, layer_forward, layer_inputs, make_inputs, random_sd,
                                      records, records_from_sd, rel_errors)

A, C, H, W = 4, 16, 32, 32


def tf32(v):
    """fp32 -> tf32 by dropping the low 13 mantissa bits (what a kind::tf32 MMA reads of an fp32 operand)."""
    return (v.float().view(torch.int32) & ~0x1FFF).view(torch.float32)


def bf16(v):
    return v.float().to(torch.bfloat16).float()


def cl_swish(seed):
    """The cluster kernel's swish: h = xhat / 2 (fp32), tanh of fp16-rounded h with an error of +-2^-11, a = h + h tanh(h)."""
    g = torch.Generator().manual_seed(seed)

    def act(xh):
        h = (xh.float() * 0.5)
        t = torch.tanh(h.half().double())
        t = (t + torch.where(torch.rand(t.shape, generator=g) < 0.5, -1.0, 1.0) * 2.0 ** -11).float()
        return (h + h * t).double()
    return act


def _model(seed=5):
    from gencomm_b200.gencomm import pack_unet
    sd = random_sd(C, seed)
    cond, x = make_inputs(seed, A, C, H, W)
    sd["conv_in.bias"] = conv_in_dc_bias(sd, cond, x)
    host, _ = pack_unet(sd, C, T_STEPS)
    return sd, host, cond, x


def _chain(sd, recs, cond, x):
    """Trace tensors (NCHW float64) and pred of one evaluation, every layer on the exact outputs of the previous ones."""
    Tn = [conv_in_forward(cond, x, sd["conv_in.weight"], sd["conv_in.bias"])[0]]
    for l in range(N_LAYERS):
        Tn.append(layer_forward(l, layer_inputs(l, Tn), recs[l])[0])
    pred = conv_out_forward(Tn[26], sd["norm_out.weight"], sd["norm_out.bias"], sd["conv_out.weight"], sd["conv_out.bias"])[0]
    return Tn, pred


def test_layer_table_reproduces_unet_forward(monkeypatch):
    sd, _, cond, x = _model()
    sd64 = {k: v.double() for k, v in sd.items()}
    emb = R.timestep_embedding
    monkeypatch.setattr(R, "timestep_embedding", lambda t, dim: emb(t, dim).double())

    def temb(t):
        e = R.timestep_embedding(torch.tensor([float(t)]), 8)
        e = F.linear(e, sd64["temb.dense.0.weight"], sd64["temb.dense.0.bias"])
        return F.linear(e * torch.sigmoid(e), sd64["temb.dense.1.weight"], sd64["temb.dense.1.bias"])
    for t in range(T_STEPS):
        _, pred = _chain(sd64, records_from_sd(sd64, t, temb), cond.double(), x.double())
        ref = R.unet_forward(torch.cat([cond, x], 1).double(), torch.full((A,), float(t)), sd64)
        assert (pred - ref).abs().max() <= 1e-12 * ref.abs().max(), t


@pytest.mark.parametrize("t", range(T_STEPS))
def test_emulations_pass_and_broken_ones_fail(t):
    sd, host, cond, x = _model()
    recs = records(host, t)
    alt = records(host, t + 1 if t + 1 < T_STEPS else t - 1)
    Tn, _ = _chain(sd, recs, cond, x)
    worst = {}
    for l, L in enumerate(LAYERS):
        ins = layer_inputs(l, Tn)
        ref, E = layer_forward(l, ins, recs[l])
        emus = {"fp32": layer_forward(l, ins, recs[l], dt=torch.float32)[0]}
        if L[0] != "down":
            emus["tf32"] = layer_forward(l, ins, recs[l], dt=torch.float32, rnd=tf32)[0]
        if L[0] == "conv":
            emus["cl"] = layer_forward(l, ins, recs[l], dt=torch.float32, rnd=tf32, act=cl_swish(l))[0]
        for arith, got in emus.items():
            e = rel_errors(got, ref, E)
            worst[arith] = max(worst.get(arith, (0, 0)), e)
            assert e[0] * SENS <= KAPPA[arith] and e[1] * SENS <= RHO[arith], (l, arith, e)
        arith = "cl" if L[0] == "conv" else ("tf32" if L[0] == "up" else "fp32")
        modes = [] if l == DC_LAYER else \
            (["halo"] if L[0] != "down" else []) + (["bands"] if L[0] == "conv" else []) + (["bias"] if L[6] else [])
        for mode in modes:
            for a in {arith, "tf32"} if L[0] == "conv" else {arith}:
                bad = rel_errors(layer_forward(l, ins, recs[l], mode=mode, rec_alt=alt[l])[0], ref, E)
                k = SENS_BANDS / SENS if mode == "bands" else 1.0
                assert bad[0] >= k * SENS * KAPPA[a] and bad[1] >= k * SENS * RHO[a], (l, mode, a, bad)
    for kind, (ref, E), got in (
            ("conv_in", conv_in_forward(cond, x, sd["conv_in.weight"], sd["conv_in.bias"]),
             conv_in_forward(cond, x, sd["conv_in.weight"], sd["conv_in.bias"], dt=torch.float32, rnd=bf16)[0]),
            ("conv_out", conv_out_forward(Tn[26], sd["norm_out.weight"], sd["norm_out.bias"], sd["conv_out.weight"],
                                          sd["conv_out.bias"]),
             conv_out_forward(Tn[26], sd["norm_out.weight"], sd["norm_out.bias"], sd["conv_out.weight"], sd["conv_out.bias"],
                              dt=torch.float32, rnd=bf16)[0])):
        e = rel_errors(got, ref, E)
        assert e[0] * SENS <= KAPPA["bf16"] and e[1] * SENS <= RHO["bf16"], (kind, e)
    print(f"\n[emulated t={t}] " + " ".join(f"{k}: max {v[0]:.2e} rms {v[1]:.2e}" for k, v in worst.items()))
