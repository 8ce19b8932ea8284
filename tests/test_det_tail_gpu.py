"""GPU parity of DownsampleConv (shrink header) and the shared detection heads (SURVEY.md 8f rank 2, first slice).

Tolerance: bf16x3 tensor-core GEMMs with fp32 accumulation (fp32-grade): max|d| <= 1e-3 * max|ref|, mean|d| <= 1e-4 *
mean|ref| against the golden outputs of the reference classes and the torch fp32 oracle.
"""
import pytest
import torch

from gencomm_b200 import DetectionHeads, DownsampleConv, synth
from oracle import ref_ops as R

pytestmark = pytest.mark.gpu
T = torch.from_numpy
DEV = "cuda"


def _close(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    d = (got - ref).abs()
    assert float(d.max()) <= 1e-3 * float(ref.abs().max()), (what, float(d.max()), float(ref.abs().max()))
    assert float(d.mean()) <= 1e-4 * float(ref.abs().mean()), (what, float(d.mean()), float(ref.abs().mean()))


def test_det_tail_matches_golden(golden_det_tail):
    g = golden_det_tail
    m = DownsampleConv({"kernal_size": [3], "stride": [2], "padding": [1], "dim": [64], "input_dim": 64})
    m.load_state_dict({k[3:]: T(v) for k, v in g.items() if k.startswith("sd/")})
    out = m.to(DEV).eval()(T(g["x"]).to(DEV))
    _close(out.cpu(), T(g["ref_out"]), "shrink")
    heads = DetectionHeads(64, 2)
    with torch.no_grad():
        for i, h in enumerate((heads.cls_head, heads.reg_head, heads.dir_head)):
            h.weight.copy_(T(g[f"head{i}/weight"])); h.bias.copy_(T(g[f"head{i}/bias"]))
    res = heads.to(DEV)(T(g["ref_out"]).to(DEV))
    for i, r in enumerate(res):
        _close(r.cpu(), T(g[f"head{i}/out"]), f"head{i}")


@pytest.mark.parametrize("cin,cout,H,W,stride,N", [(384, 128, 128, 256, 2, 1), (256, 128, 64, 128, 1, 2), (64, 256, 8, 48, 1, 1),
                                                   (384, 256, 128, 256, 2, 8)])
def test_downsample_conv_matches_oracle(cin, cout, H, W, stride, N):
    """The GenComm stage-1 shrink header (384 -> 128, stride 2, 128x256 -> 64x128), a stride-1 header, a 256-column
    case with rows that are not a multiple of the tile, and the configs[3] header (384 -> 256) over 8 agents: 512 tiles,
    three or more per CTA pair of the multicast kernel."""
    torch.manual_seed(cin + H)
    cfg = {"kernal_size": [3], "stride": [stride], "padding": [1], "dim": [cout], "input_dim": cin}
    m = DownsampleConv(cfg).eval()
    x = synth.bev_features(55, N, cin, H, W)
    ref = R.downsample_conv(x, {k: v.detach() for k, v in m.state_dict().items()}, [stride])
    out = m.to(DEV)(x.to(DEV)).cpu()
    _close(out, ref, "shrink")


def test_det_heads_match_oracle_and_errors():
    """C = 128 (OPV2V-H) over 3 frames and C = 256 (V2X-Real) over 8 frames (512 tiles: three or more per CTA)."""
    for C, B in ((128, 3), (256, 8)):
        torch.manual_seed(2)
        heads = DetectionHeads(C, 2).eval()
        x = synth.bev_features(66, B, C, 64, 128)
        ref = R.det_heads(x, *[t.detach() for h in (heads.cls_head, heads.reg_head, heads.dir_head) for t in (h.weight, h.bias)])
        got = heads.to(DEV)(x.to(DEV))
        for name, a, b in zip(("cls", "reg", "dir"), got, ref):
            _close(a.cpu(), b, f"{name} C={C}")
    with pytest.raises(RuntimeError, match="multiple of 128"):
        heads(torch.zeros(1, 128, 3, 10, device=DEV))
    bad = DownsampleConv({"kernal_size": [3], "stride": [1], "padding": [1], "dim": [64], "input_dim": 48}).to(DEV)
    with pytest.raises(RuntimeError, match="multiples of 64"):
        bad(torch.zeros(1, 48, 8, 16, device=DEV))
