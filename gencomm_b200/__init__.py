"""gencomm_b200 -- B200-native (sm_100a) implementation of GenComm's per-frame hot path.

    points -> voxelize -> PillarVFE -> PointPillarScatter -> BEV canvas
    BEV features -> warp to ego (affine_grid + grid_sample) + regroup + Max/Att fusion
    GenComm conditional-diffusion sampler (DiffusionUNet denoiser)

Hand-written CUDA behind a C ABI (include/gencomm_b200.h, csrc/), loaded through ctypes; the
classes in ``gencomm_b200.modules`` carry the reference's operator names and signatures.
"""
from . import _lib, ops, synth  # noqa: F401
from .modules import (AttFusion, BEVFeatureInput, MaxFusion, PFNLayer, PillarVFE, PointPillar, PointPillarScatter,  # noqa: F401
                      SpVoxelPreprocessor, normalize_pairwise_tfm, regroup, warp_affine_simple, warp_feature)

from .gencomm import Config, DiffusionUNet, GenComm  # noqa: F401
from .message_extractor import BEVDeformableExtractor, MessageExtractorv2  # noqa: F401
from .enhancer import Enhancer  # noqa: F401
from .det_tail import DetectionHeads, DoubleConv, DownsampleConv  # noqa: F401
from .backbone import BaseBEVBackbone  # noqa: F401
from .postprocess import VoxelPostprocessor  # noqa: F401
from .lss import VoxelPooling, gen_dx_bx, voxel_pooling  # noqa: F401
from . import eval_utils  # noqa: F401
from .eval_utils import DetectionEvaluator, caluclate_tp_fp  # noqa: F401

from .heter_model_baseline import HeterModelBaseline  # noqa: F401
from .heter_model_baseline_w_gencomm_stage1 import HeterModelBaselineWGenComm  # noqa: F401
from .heter_model_baseline_w_gencomm_stage2 import HeterModelBaselineWDiffCommStage2  # noqa: F401


def create_model(hypes):
    """``train_utils.create_model`` (tools/train_utils.py:255-288) over this package: resolves
    ``gencomm_b200.<core_method>`` and the class whose lower-cased name is ``core_method`` without underscores."""
    import importlib
    name = hypes['model']['core_method']
    try:
        lib = importlib.import_module(f"{__name__}.{name}")
    except ModuleNotFoundError as e:
        raise NotImplementedError(f"gencomm_b200 has no model {name!r} (HeterModelBaseline and the GenComm stage 1 / "
                                  "stage 2 detectors only)") from e
    target = name.replace('_', '').lower()
    for attr, cls in lib.__dict__.items():
        if attr.lower() == target:
            return cls(hypes['model']['args'])
    # Reference quirk: the shipped yamls name the FILE (heter_model_baseline_w_gencomm_stage1 / _stage2) while the classes
    # are called HeterModelBaselineWGenComm / HeterModelBaselineWDiffCommStage2, which the name rule above cannot match.
    # Fall back to the one model class the module itself defines.
    own = [c for c in lib.__dict__.values() if isinstance(c, type) and c.__module__ == lib.__name__
           and not c.__name__.startswith('_')]
    if len(own) == 1:
        return own[0](hypes['model']['args'])
    raise NotImplementedError(f"no class matching {target!r} in {lib.__name__}")


__version__ = "0.1.0"
