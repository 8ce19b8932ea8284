"""GPU parity of the Enhancer (SURVEY.md 8f rank 1) against the golden vectors of the reference class and the oracle.

Tolerance: the three dense layers run as bf16x3 tensor-core GEMMs (fp32-grade), the rest is fp32 in a different summation
order than torch: max|d| <= 1e-3 * max|ref| and mean|d| <= 1e-4 * mean|ref| (stated here; measured ~1e-5 / 1e-6).
"""
import pytest
import torch

from gencomm_b200 import Enhancer, synth
from oracle import ref_ops as R

pytestmark = pytest.mark.gpu
T = torch.from_numpy
DEV = "cuda"


def _close(got, ref, what):
    d = (got - ref).abs()
    assert float(d.max()) <= 1e-3 * float(ref.abs().max()), (what, float(d.max()), float(ref.abs().max()))
    assert float(d.mean()) <= 1e-4 * float(ref.abs().mean()), (what, float(d.mean()), float(ref.abs().mean()))


def test_enhancer_matches_golden(golden_enhancer):
    g = golden_enhancer
    x = T(g["x"])
    model = Enhancer(x.shape[1], [8, 8], 4)
    model.load_state_dict({k[3:]: T(v) for k, v in g.items() if k.startswith("sd/")}, strict=False)
    model = model.to(DEV).eval()
    out = model(x.to(DEV), T(g["affine"]).to(DEV), T(g["record_len"]).to(DEV)).cpu()
    _close(out, T(g["ref_out"]), "enhancer")


@pytest.mark.parametrize("C,H,W,N", [(128, 64, 128, 2), (256, 8, 48, 2), (128, 2, 64, 1), (256, 64, 128, 8)])
def test_enhancer_matches_oracle(C, H, W, N):
    """OPV2V-H (C=128, 64x128) and V2X-Real (C=256) shapes, rows that are not a multiple of the 128-pixel tile, and
    C=256 at 64x128 over 8 agents (the GEMMs on CTA pairs, three or more tiles per CTA), against the oracle restatement on
    the same seeded inputs and randomised LayerNorm / bias parameters."""
    torch.manual_seed(C + W)
    model = Enhancer(C, [8, 8], 4).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "norm" in name or "bn1" in name:
                p.add_(0.2 * torch.randn_like(p))
            elif name.endswith(".bias"):
                p.add_(0.1 * torch.randn_like(p))
    x = synth.bev_features(91, N, C, H, W)
    x[-1, :, :, W // 2:] = 0.0
    ref = R.enhancer(x, {k: v.detach() for k, v in model.state_dict().items()})
    out = model.to(DEV)(x.to(DEV)).cpu()
    _close(out, ref, "enhancer")


def test_enhancer_argument_errors():
    with pytest.raises(RuntimeError, match="128 or 256"):
        Enhancer(64, [8, 8], 4).to(DEV)(torch.zeros(1, 64, 4, 32, device=DEV))
    m = Enhancer(128, [8, 8], 4).to(DEV)
    with pytest.raises(RuntimeError, match="multiple of 128"):
        m(torch.zeros(1, 128, 3, 10, device=DEV))
    assert m(torch.zeros(0, 128, 4, 32, device=DEV)).shape == (0, 128, 4, 32)
