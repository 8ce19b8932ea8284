"""GPU tests of HeterModelBaseline -- the heterogeneous intermediate-fusion detector without GenComm.

Bit for bit against the GenComm detectors: a GenComm detector and the baseline are built from ONE synth.fill_state_dict
fill, so every module they share carries the same weights.  The baseline's fusion input must then equal the GenComm
detector's ``gt_feature`` exactly (same encoder -> backbone -> shrink header kernels, camera padding and per-agent
re-assembly), and its heads must equal the GenComm detector's own ``fusion_net`` (+ ``shrink_conv``) + heads applied to
that ``gt_feature`` exactly.

Against the oracle: the heads against the composition of the oracle/ref_ops restatements without the GenComm stages (PFN
-> scatter -> BaseBEVBackbone -> DownsampleConv -> warp + Att/Max fusion -> shrink_conv -> heads, fp32 torch on the
host).  The convolutions run as bf16x3 tcgen05 GEMMs (fp32-grade: three bf16 products recover the fp32 operands to about
2^-16 relative); through the 17-layer backbone, the shrink header and the heads that gives the bound the GenComm detector
states for its ``gt_feature`` (tests/test_heter_model_gpu.py): max|d| <= 1e-3 * max|ref|, mean|d| <= 3e-4 * mean|ref|.
Warp + fusion adds <= 1e-5 (tests/test_warp_fuse_gpu.py).
"""
import numpy as np
import pytest
import torch

import gencomm_b200 as G
from gencomm_b200 import synth
from oracle import gen_golden
from oracle import ref_ops as R

pytestmark = pytest.mark.gpu
T = torch.from_numpy
DEV = "cuda"
RAGGED = [1, 3, 5]                       # agents per frame
RAGGED_SEED, WSEED = 4500, 29
TMAX, TMEAN = 1e-3, 3e-4
EXTRAS = {"supervise_single": True, "in_head_single": 128,
          "shrink_header": {"kernal_size": [3], "stride": [1], "padding": [1], "dim": [128], "input_dim": 128}}


@pytest.fixture(scope="module")
def ragged_inputs():
    """Three frames of 1, 3 and 5 LiDAR agents: voxel tensors, the same clouds as raw points, poses, record_len."""
    clouds, pairwise = synth.heter_frames(RAGGED_SEED, RAGGED, gen_golden.HETER_POINTS)
    voxels = R.collate_voxels([R.voxelize(c, synth.OPV2V_H_RANGE, [0.4, 0.4, 4.0]) for c in clouds])
    off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int32)
    points = {"points": T(np.concatenate(clouds)), "point_offsets": T(off), "max_agent_points": max(len(c) for c in clouds)}
    return voxels, points, T(pairwise), torch.tensor(RAGGED, dtype=torch.int64)


def _data(inputs, kind):
    voxels, points, pairwise, record_len = inputs
    inp = voxels if kind == "voxels" else points
    return {"inputs_m1": {k: v.to(DEV) if torch.is_tensor(v) else v for k, v in inp.items()},
            "agent_modality_list": ["m1"] * int(record_len.sum()), "pairwise_t_matrix": pairwise.to(DEV),
            "record_len": record_len.to(DEV)}


def _pair(gen_args, gen_cls=G.HeterModelBaselineWGenComm, seed=WSEED):
    """(GenComm detector, baseline) on the device, from one weight fill."""
    gen = gen_cls(gen_args)
    sd = synth.fill_state_dict(gen.state_dict(), seed)
    gen.load_state_dict(sd)
    base = G.HeterModelBaseline(synth.without_gencomm(gen_args))
    assert base.load_state_dict(sd, strict=False).missing_keys == []
    return gen.to(DEV).eval(), base.to(DEV).eval()


def _run_baseline(base, data):
    """(output dict, the per-agent features the baseline hands to its fusion_net)."""
    seen = []
    hook = base.fusion_net.register_forward_pre_hook(lambda _m, inp: seen.append(inp[0].clone()))
    try:
        out = base(dict(data))
    finally:
        hook.remove()
    assert len(seen) == 1
    return out, seen[0]


@torch.no_grad()
def _gencomm_tail(gen, gt_feature, data):
    """The GenComm detector's own fusion_net -> shrink_conv -> heads on its gt_feature."""
    affine = G.normalize_pairwise_tfm(data["pairwise_t_matrix"], gen.H, gen.W, 1)
    fused = gen.fusion_net(gt_feature, data["record_len"], affine)
    if gen.shrink_flag:
        fused = gen.shrink_conv(fused)
    return dict(zip(("cls_preds", "reg_preds", "dir_preds"), gen._run_heads(fused)))


def _check_bit_exact(gen, base, data, extras):
    ref = gen(dict(data))
    out, fused_in = _run_baseline(base, data)
    heads = {"cls_preds", "reg_preds", "dir_preds"}
    single = {k + "_single" for k in heads}
    assert set(out) == heads | (single if extras else set())
    assert torch.equal(fused_in, ref["gt_feature"])
    for k, v in _gencomm_tail(gen, ref["gt_feature"], data).items():
        assert torch.equal(out[k], v), k
    for k in (single if extras else ()):
        assert torch.equal(out[k], ref[k]), k
    return out, fused_in


@pytest.mark.parametrize("fusion,kind,extras", [("att", "voxels", False), ("max", "points", False),
                                                ("att", "points", True), ("max", "voxels", True)],
                         ids=["att-voxels", "max-points", "att-points-single-shrink", "max-voxels-single-shrink"])
def test_baseline_equals_stage1_components(ragged_inputs, fusion, kind, extras):
    """Ragged record_len (1, 3, 5 agents); ``extras``: supervise_single heads and a shrink_conv after the fusion."""
    args = synth.gencomm_stage1_args(fusion)
    if extras:
        args.update(EXTRAS)
    gen, base = _pair(args)
    out, _ = _check_bit_exact(gen, base, _data(ragged_inputs, kind), extras)
    assert out["cls_preds"].shape == (3, 2, 64, 128) and out["reg_preds"].shape == (3, 14, 64, 128)
    if extras:
        assert out["cls_preds_single"].shape == (9, 2, 64, 128)


def test_lidar_camera_baseline_equals_stage2_components(heter2_inputs):
    """LiDAR (m1) + camera (m2) agents interleaved over 3 + 2 agents: the camera BEV feature through its backbone and
    shrink header, zero-padded to the LiDAR extent, re-assembled in agent order -- equal to the stage-2 detector's."""
    voxels, bev, pairwise, record_len, _, _ = heter2_inputs
    data = {"inputs_m1": {k: v.to(DEV) for k, v in voxels.items()}, "inputs_m2": {"bev_feature": bev.to(DEV)},
            "agent_modality_list": list(gen_golden.HETER2_MODALITIES), "pairwise_t_matrix": pairwise.to(DEV),
            "record_len": record_len.to(DEV)}
    gen, base = _pair(synth.gencomm_stage2_hetero_args("att"), G.HeterModelBaselineWDiffCommStage2, gen_golden.HETER2_WSEED)
    _, fused_in = _check_bit_exact(gen, base, data, False)
    assert fused_in.shape == (5, 128, 64, 128)
    for a in (1, 4):   # the camera agents carry exact zeros outside the central 64 columns
        assert float(fused_in[a][:, :, :32].abs().max()) == 0.0 and float(fused_in[a][:, :, 96:].abs().max()) == 0.0


def _oracle(sd, args, voxels, pairwise, record_len):
    """HeterModelBaseline.forward restated from oracle/ref_ops: heter_gencomm_forward without the message extractor, the
    sampler and the Enhancer, plus the optional shrink_conv and supervise_single heads."""
    sub = lambda prefix: {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    setting = args["m1"]
    enc, rng = setting["encoder_args"], args["lidar_range"]
    affine = R.normalize_pairwise_tfm(pairwise, rng[4] - rng[1], rng[3] - rng[0], 1)
    p = sub("encoder_m1.pillar_vfe.pfn_layers.0.")
    pf = R.pillar_vfe(voxels["voxel_features"], voxels["voxel_num_points"], voxels["voxel_coords"], p["linear.weight"],
                      p["norm.weight"], p["norm.bias"], p["norm.running_mean"], p["norm.running_var"],
                      enc["voxel_size"], enc["lidar_range"])
    g = R.grid_size(enc["lidar_range"], enc["voxel_size"])
    x = R.scatter(pf, voxels["voxel_coords"], int(g[0]), int(g[1]), int(record_len.sum()))
    b = setting["backbone_args"]
    x = R.bev_backbone(x, sub("backbone_m1."), b["layer_nums"], b["layer_strides"], b["upsample_strides"])
    x = R.downsample_conv(x, sub("shrinker_m1."), setting["shrink_header"]["stride"])
    heads = lambda t, s: R.det_heads(t, *(sd[f"{h}_head{s}.{w}"] for h in ("cls", "reg", "dir") for w in ("weight", "bias")))
    out = {}
    if args.get("supervise_single"):
        out.update(zip(("cls_preds_single", "reg_preds_single", "dir_preds_single"), heads(x, "_single")))
    fused = (R.att_fusion if args["fusion_method"] == "att" else R.max_fusion)(x, record_len, affine)
    if "shrink_header" in args:
        fused = R.downsample_conv(fused, sub("shrink_conv."), args["shrink_header"]["stride"])
    out.update(zip(("cls_preds", "reg_preds", "dir_preds"), heads(fused, "")))
    return out


@pytest.mark.parametrize("fusion,extras", [("att", False), ("max", True)], ids=["att", "max-single-shrink"])
def test_baseline_matches_oracle(heter_inputs, ragged_inputs, fusion, extras):
    """att: the 2 + 1 agents of tests/golden/heter_model.npz; max: the ragged 1 + 3 + 5 agents with supervise_single and
    shrink_conv.  Bound in the module docstring."""
    args = synth.heter_baseline_args(fusion)
    if extras:
        args.update(EXTRAS)
        voxels, _, pairwise, record_len = ragged_inputs
    else:
        voxels, pairwise, record_len, _, _ = heter_inputs
    m = G.HeterModelBaseline(args)
    m.load_state_dict(synth.fill_state_dict(m.state_dict(), WSEED))
    m = m.to(DEV).eval()
    out = m({"inputs_m1": {k: v.to(DEV) for k, v in voxels.items()}, "agent_modality_list": ["m1"] * int(record_len.sum()),
             "pairwise_t_matrix": pairwise.to(DEV), "record_len": record_len.to(DEV)})
    ref = _oracle({k: v.cpu() for k, v in m.state_dict().items()}, args, voxels, pairwise, record_len)
    assert set(out) == set(ref)
    for k in ref:
        got = out[k].cpu()
        assert got.shape == ref[k].shape, (k, got.shape, ref[k].shape)
        d = (got - ref[k]).abs()
        emax, emean = float(d.max()) / float(ref[k].abs().max()), float(d.mean()) / float(ref[k].abs().mean())
        print(f"{fusion} {k}: max {emax:.2e} mean {emean:.2e}")
        assert emax <= TMAX and emean <= TMEAN, (k, emax, emean)


TORCH_GEMM_OPS = ("aten::conv", "aten::_conv", "aten::cudnn", "aten::mkldnn", "aten::mm", "aten::addmm", "aten::bmm",
                  "aten::baddbmm", "aten::matmul", "aten::linear", "aten::einsum", "aten::_scaled_mm", "aten::addmv")
VENDOR_KERNELS = ("gemm", "conv", "xmma", "cudnn", "cutlass", "cublas", "nvjet", "winograd", "sm90_", "sm100_")


def test_baseline_forward_runs_no_torch_conv_or_matmul(ragged_inputs):
    """torch.profiler over two forwards from raw points (the first packs the weights): no torch convolution / matrix
    product op, no vendor GEMM or convolution kernel; the pillar, convolution, fusion and pose kernels are this package's.
    After the first call the forward does not synchronise with the host."""
    from torch.profiler import ProfilerActivity, profile
    m = G.HeterModelBaseline(synth.heter_baseline_args("att"))
    m.load_state_dict(synth.fill_state_dict(m.state_dict(), WSEED))
    m = m.to(DEV).eval()
    data = _data(ragged_inputs, "points")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            m(dict(data))
            torch.cuda.synchronize()
    cpu_ops = {e.name for e in prof.events() if e.device_type.name == "CPU"}
    kernels = {e.name.removeprefix("void ").split("(")[0].split("<")[0] for e in prof.events()
               if e.device_type.name == "CUDA"}
    assert not {n for n in cpu_ops if n.startswith(TORCH_GEMM_OPS)}
    own = {n.split("::")[-1] for n in kernels if n.split("::")[-1].startswith("k_")}
    other = {n for n in kernels if not n.split("::")[-1].startswith("k_")}
    assert not {n for n in other if any(s in n.lower() for s in VENDOR_KERNELS)}, sorted(other)
    assert {"k_pillar_build", "k_conv_tma", "k_normalize_tfm"} <= own and any("fuse" in n for n in own), sorted(own)
    torch.cuda.set_sync_debug_mode("error")
    try:
        m(dict(data))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
