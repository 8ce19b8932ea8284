"""HeterModelBaseline (heterogeneous intermediate fusion without GenComm) on the host: model resolution, state_dict keys
against the stage-1 / stage-2 GenComm detectors, checkpoint loading, refusals."""
import pytest
import torch

import gencomm_b200 as G
from gencomm_b200 import synth

GENCOMM_PREFIXES = ("gencomm.", "enhancer.", "message_extractor_")


def _without_gencomm_keys(sd):
    return [k for k in sd if not k.startswith(GENCOMM_PREFIXES)]


def test_create_model_resolves_heter_model_baseline():
    m = G.create_model({"model": {"core_method": "heter_model_baseline", "args": synth.heter_baseline_args("max")}})
    assert type(m) is G.HeterModelBaseline and isinstance(m.fusion_net, G.MaxFusion) and not m.training
    m = G.create_model({"model": {"core_method": "heter_model_baseline", "args": synth.heter_baseline_args("att")}})
    assert isinstance(m.fusion_net, G.AttFusion)
    for name in ("gencomm", "enhancer", "message_extractor_m1", "missing_message"):
        assert not hasattr(m, name), name
    assert isinstance(G.HeterModelBaselineWGenComm(synth.gencomm_stage1_args("att")), G.HeterModelBaseline)


def test_baseline_args_drop_only_the_gencomm_blocks():
    s1, b = synth.gencomm_stage1_args("att"), synth.heter_baseline_args("att")
    assert set(s1) - set(b) == {"gencomm", "enhancer", "message_extractor"} and set(b) <= set(s1)
    s2, bh = synth.gencomm_stage2_hetero_args("max"), synth.heter_baseline_hetero_args("max")
    assert set(s2) - set(bh) == {"diffcomm", "enhancer", "message_extractor"} and bh["m2"]["sensor_type"] == "camera"


@pytest.mark.parametrize("variant", ["lidar", "lidar_camera", "single_heads_shrink_conv"])
def test_state_dict_is_the_gencomm_detectors_minus_gencomm(variant):
    """Same keys, in the same order, with the same shapes as the GenComm detector built from the same arguments, minus
    the GenComm modules; the GenComm detector registers those where the reference does (sampler first, each message
    extractor after its shrink header, Enhancer after the heads)."""
    if variant == "lidar_camera":
        gen, base = G.HeterModelBaselineWDiffCommStage2(synth.gencomm_stage2_hetero_args("att")), \
            G.HeterModelBaseline(synth.heter_baseline_hetero_args("att"))
    else:
        a = synth.gencomm_stage1_args("att")
        if variant == "single_heads_shrink_conv":
            a.update(supervise_single=True, in_head_single=128,
                     shrink_header={"kernal_size": [3], "stride": [1], "padding": [1], "dim": [128], "input_dim": 128})
        gen, base = G.HeterModelBaselineWGenComm(a), G.HeterModelBaseline(synth.without_gencomm(a))
    gsd, bsd = gen.state_dict(), base.state_dict()
    assert list(bsd) == _without_gencomm_keys(gsd)
    assert all(bsd[k].shape == gsd[k].shape for k in bsd)
    keys = list(gsd)
    n_sampler = sum(k.startswith("gencomm.") for k in keys)
    assert all(k.startswith("gencomm.") for k in keys[:n_sampler])
    for m in gen.modality_name_list:
        first_me = next(i for i, k in enumerate(keys) if k.startswith(f"message_extractor_{m}."))
        assert first_me == 1 + max(i for i, k in enumerate(keys) if k.startswith(f"shrinker_{m}.")), m
    assert all(k.startswith("enhancer.") for k in keys[keys.index("dir_head.bias") + 1:])
    if variant == "single_heads_shrink_conv":
        assert "cls_head_single.weight" in bsd and "shrink_conv.layers.0.double_conv.0.weight" in bsd


def test_stage1_checkpoint_loads_with_nothing_missing():
    s1 = G.HeterModelBaselineWGenComm(synth.gencomm_stage1_args("att"))
    ckpt = synth.fill_state_dict(s1.state_dict(), 5)
    base = G.HeterModelBaseline(synth.heter_baseline_args("att"))
    res = base.load_state_dict(ckpt, strict=False)
    assert res.missing_keys == []
    assert sorted(res.unexpected_keys) == sorted(k for k in ckpt if k.startswith(GENCOMM_PREFIXES))
    for k, v in base.state_dict().items():
        assert torch.equal(v, ckpt[k]), k


def _refusal(cls, args):
    with pytest.raises(NotImplementedError) as e:
        cls(args)
    return str(e.value)


@pytest.mark.parametrize("case", ["compressor", "fusion_method", "encoder"])
def test_refusals_match_stage1(case):
    def args(base):
        a = synth.heter_baseline_args("att") if base else synth.gencomm_stage1_args("att")
        if case == "compressor":
            a["compressor"] = {"input_dim": 128, "compress_ratio": 32}
        elif case == "fusion_method":
            a["fusion_method"] = "v2xvit"
        else:
            a["m3"] = dict(a["m1"], core_method="second")
        return a
    msg = _refusal(G.HeterModelBaseline, args(True))
    assert msg == _refusal(G.HeterModelBaselineWGenComm, args(False))
    assert {"compressor": "NaiveCompressor", "fusion_method": "fusion_method", "encoder": "LiDAR"}[case] in msg


def test_baseline_is_inference_only():
    m = G.HeterModelBaseline(synth.heter_baseline_args("att"))
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m({})
