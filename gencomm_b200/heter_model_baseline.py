"""Drop-in ``HeterModelBaseline`` -- heterogeneous intermediate fusion without GenComm, assembled from the B200 operators.

Mirrors ``opencood/models/heter_model_baseline.py:27-253`` (BASELINE.json configs 1-2): every agent shares its full BEV
feature; the features are warped to the ego and fused with Max / Att, then the optional ``shrink_conv`` and the heads run.
It is the stage-1 GenComm detector without the message extractor, the sampler and the Enhancer -- the comparison every
GenComm evaluation runs -- and ``HeterModelBaselineWGenComm`` (``heter_model_baseline_w_gencomm_stage1.py``) extends this
class with them.  Same constructor argument dict (``model.args``), same sub-module names (``encoder_m1``, ``backbone_m1``,
``shrinker_m1``, ``fusion_net``, ``shrink_conv``, ``cls_head`` / ``reg_head`` / ``dir_head``, the ``_single`` heads) so a
reference checkpoint loads with ``load_state_dict`` (a GenComm checkpoint loads with ``strict=False``: its extra keys are
the GenComm modules), same ``forward(data_dict)`` contract:

    data_dict: inputs_m{k} {voxel_features, voxel_coords, voxel_num_points}, agent_modality_list, pairwise_t_matrix
               [B,L,L,4,4] f64, record_len [B]
    returns:   cls_preds, reg_preds, dir_preds (+ cls_preds_single, reg_preds_single, dir_preds_single with supervise_single)

Every stage runs a hand-written sm_100a kernel through the C ABI: voxels -> PillarVFE -> scatter canvas (pillars.cu),
BaseBEVBackbone + shrink header (tcgen05 implicit GEMMs), warp + Max/Att fusion, detection heads.  Inference only; no CPU
path; the forward never synchronises with the host.

Scope: LiDAR ``point_pillar`` modalities, camera ``lift_splat_shoot`` modalities through their BEV feature
(``data_dict['inputs_m{k}']['bev_feature']`` or ``set_encoder``; see ``modules.BEVFeatureInput``) and ``fusion_method``
max / att.  The other encoders, the other fusion networks and the training-only compressor raise ``NotImplementedError`` at
construction.  Extension (ignored by the reference): ``data_dict['inputs_m{k}']`` may carry raw ``points`` +
``point_offsets`` (see ``modules.PointPillar``).
"""
from collections import Counter, OrderedDict

import torch
import torch.nn as nn

from .backbone import BaseBEVBackbone
from .det_tail import DetectionHeads, DownsampleConv
from .modules import AttFusion, BEVFeatureInput, MaxFusion, PointPillar, center_crop, normalize_pairwise_tfm

_ENCODERS = {("lidar", "pointpillar"): PointPillar, ("camera", "liftsplatshoot"): BEVFeatureInput}


class _HeadsMixin:
    """The three 1x1 heads keep their reference names / state_dict keys; they are evaluated as one GEMM."""

    def _run_heads(self, x, suffix=""):
        key = "_heads" + suffix
        heads = getattr(self, key, None)
        if heads is None:
            heads = DetectionHeads.__new__(DetectionHeads)
            nn.Module.__init__(heads)
            heads.cls_head = getattr(self, "cls_head" + suffix)
            heads.reg_head = getattr(self, "reg_head" + suffix)
            heads.dir_head = getattr(self, "dir_head" + suffix)
            heads._key, heads._blobs = None, None
            object.__setattr__(self, key, heads)     # not registered: the convs stay owned by this module
        return heads(x)


class HeterModelBaseline(_HeadsMixin, nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self._add_sampler(args)
        self.modality_name_list = [x for x in args.keys() if x.startswith("m") and x[1:].isdigit()]
        self.ego_modality = args['ego_modality']
        self.cav_range = args['lidar_range']
        self.sensor_type_dict = OrderedDict()

        for modality_name in self.modality_name_list:
            setting = args[modality_name]
            self.sensor_type_dict[modality_name] = setting['sensor_type']
            target = setting['core_method'].replace('_', '').lower()
            if (setting['sensor_type'], target) not in _ENCODERS:
                raise NotImplementedError(
                    f"gencomm_b200: modality {modality_name} ({setting['sensor_type']}/{setting['core_method']}) -- LiDAR "
                    "point_pillar encoders and camera lift_splat_shoot BEV features are on the B200 hot path")
            setattr(self, f"encoder_{modality_name}", _ENCODERS[(setting['sensor_type'], target)](setting['encoder_args']))
            if setting['sensor_type'] == 'camera':      # heter_model_baseline_w_gencomm_stage1.py:88-92
                grid = setting['camera_mask_args']['grid_conf']
                setattr(self, f"crop_ratio_W_{modality_name}", self.cav_range[3] / grid['xbound'][1])
                setattr(self, f"crop_ratio_H_{modality_name}", self.cav_range[4] / grid['ybound'][1])
            setattr(self, f"depth_supervision_{modality_name}", False)
            if setting['backbone_args'] == 'identity':
                setattr(self, f"backbone_{modality_name}", nn.Identity())
            else:
                setattr(self, f"backbone_{modality_name}",
                        BaseBEVBackbone(setting['backbone_args'], setting['backbone_args'].get('inplanes', 64)))
            setattr(self, f"shrinker_{modality_name}", DownsampleConv(setting['shrink_header']))
            self._add_message_extractor(modality_name, args)

        # metric extents for the pose normalisation (heter_model_baseline.py:87-89)
        self.H = self.cav_range[4] - self.cav_range[1]
        self.W = self.cav_range[3] - self.cav_range[0]
        self.fake_voxel_size = 1
        self.gmatch = bool(args.get('gmatch', False))
        self.num_class = args['num_class'] if "num_class" in args else 1
        anchors, bins = args['anchor_number'], args['dir_args']['num_bins']

        self.supervise_single = bool(args.get("supervise_single", False))
        if self.supervise_single:
            c = args['in_head_single']
            self.cls_head_single = nn.Conv2d(c, anchors * self.num_class * self.num_class, kernel_size=1)
            self.reg_head_single = nn.Conv2d(c, anchors * 7 * self.num_class, kernel_size=1)
            self.dir_head_single = nn.Conv2d(c, anchors * bins, kernel_size=1)

        if args['fusion_method'] == "max":
            self.fusion_net = MaxFusion()
        elif args['fusion_method'] == "att":
            self.fusion_net = AttFusion(args['att']['feat_dim'])
        else:
            raise NotImplementedError(f"gencomm_b200: fusion_method {args['fusion_method']!r} -- max and att are on the "
                                      "B200 hot path (SURVEY.md 8a rows a8/a9)")

        self.shrink_flag = 'shrink_header' in args
        if self.shrink_flag:
            self.shrink_conv = DownsampleConv(args['shrink_header'])

        self.cls_head = nn.Conv2d(args['in_head'], anchors * self.num_class * self.num_class, kernel_size=1)
        self.reg_head = nn.Conv2d(args['in_head'], 7 * anchors * self.num_class, kernel_size=1)
        self.dir_head = nn.Conv2d(args['in_head'], bins * anchors, kernel_size=1)
        self._add_enhancer(args)

        self.compress = False
        if 'compressor' in args:
            raise NotImplementedError("gencomm_b200: the NaiveCompressor is a training-only add-on (…_stage1.py:152-158)")
        self.eval()

    # The GenComm detectors add their modules through these hooks, at the places where the reference constructs them, so
    # that their state_dict keys keep the reference's order and their default initialisation draws the same random numbers.
    def _add_sampler(self, args):
        pass

    def _add_message_extractor(self, modality_name, args):
        pass

    def _add_enhancer(self, args):
        pass

    def invalidate(self):
        """Drop every packed-weight cache of the detector (after in-place parameter writes through ``p.data``)."""
        for m in self.modules():
            if m is not self and hasattr(m, "invalidate"):
                m.invalidate()
        for key in ("_heads", "_heads_single"):
            h = getattr(self, key, None)
            if h is not None:
                h.invalidate()

    def _load_from_state_dict(self, *args, **kwargs):
        for key in ("_heads", "_heads_single"):      # the fused-heads helper is not a registered sub-module
            h = getattr(self, key, None)
            if h is not None:
                h.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def set_encoder(self, modality_name, module):
        """Plug in an encoder for a modality (e.g. the reference's own ``LiftSplatShoot`` instance): it is called as
        ``module(data_dict, modality_name)`` like heter_encoders' classes and must return the BEV feature on the device."""
        setattr(self, f"encoder_{modality_name}", module)

    def _encode(self, data_dict, after_encoder=None):
        """Yields ``(modality, feature [n_m, C, H, W])`` for every modality present in ``agent_modality_list``, in the
        order of ``modality_name_list``: encoder -> backbone -> shrink header (heter_model_baseline_w_gencomm_stage1.py:
        185-194).  ``after_encoder()``, if given, is called between the encoder and the backbone of each modality."""
        counts = Counter(data_dict['agent_modality_list'])
        for m in self.modality_name_list:
            if m not in counts:
                continue
            inp = data_dict[f'inputs_{m}']
            if 'points' not in inp and 'batch_size' not in inp:
                # the agent count is known on the host: spares PointPillarScatter's `.item()` sync (point_pillar_scatter.py:45)
                data_dict = dict(data_dict)
                data_dict[f'inputs_{m}'] = dict(inp, batch_size=counts[m])
            encoder, backbone = getattr(self, f"encoder_{m}"), getattr(self, f"backbone_{m}")
            shrinker = getattr(self, f"shrinker_{m}")
            # raw points straight into this package's backbone: the canvas is written as its operand planes
            planes_in = isinstance(encoder, PointPillar) and isinstance(backbone, BaseBEVBackbone) and 'points' in inp
            try:
                if planes_in:
                    encoder.emit_planes = True
                feature = encoder(data_dict, m)
            finally:
                if planes_in:
                    encoder.emit_planes = False
            if after_encoder is not None:
                after_encoder()
            if not isinstance(backbone, nn.Identity):
                # the shrink header follows directly: the deblocks write its operand planes, no NCHW fp32 round trip
                fused = isinstance(backbone, BaseBEVBackbone) and isinstance(shrinker, DownsampleConv)
                try:
                    if fused:
                        backbone.emit_planes = True
                    feature = backbone({"spatial_features": feature})['spatial_features_2d']
                finally:
                    if fused:
                        backbone.emit_planes = False
            feature = shrinker(feature)       # drops the backbone output before the caller's loop body runs
            yield m, feature

    def _pad_to_lidar(self, m, x):
        """Camera feature maps cover the camera grid only: zero-pad them to the LiDAR extent
        (heter_model_baseline_w_gencomm_stage1.py:199-213)."""
        if self.sensor_type_dict[m] != "camera":
            return x
        h, w = x.shape[-2:]
        return center_crop(x, int(h * getattr(self, f"crop_ratio_H_{m}")), int(w * getattr(self, f"crop_ratio_W_{m}")))

    @staticmethod
    def _per_agent(maps, agent_modality_list):
        """Restore the per-agent order from the per-modality batches ``maps[m] [n_m, ...]``
        (heter_model_baseline_w_gencomm_stage1.py:215-228)."""
        if len(maps) == 1 and all(a == agent_modality_list[0] for a in agent_modality_list):
            x = maps[agent_modality_list[0]]
            if x.shape[0] != len(agent_modality_list):
                raise ValueError("agent_modality_list does not match the number of encoded agents")
            return x
        seen = dict.fromkeys(maps, 0)
        per_agent = []
        for m in agent_modality_list:
            per_agent.append(maps[m][seen[m]])
            seen[m] += 1
        return torch.stack(per_agent)

    def _single_preds(self, x):
        """The per-agent heads of ``supervise_single`` on the per-agent features (an empty dict without them)."""
        if not self.supervise_single:
            return {}
        c, r, d = self._run_heads(x, "_single")
        return {'cls_preds_single': c, 'reg_preds_single': r, 'dir_preds_single': d}

    def _detect(self, x, record_len, affine_matrix):
        """fusion_net -> shrink_conv (if configured) -> heads on the per-agent features ``x [ΣN, C, H, W]``."""
        fused_feature = self.fusion_net(x, record_len, affine_matrix)
        if self.shrink_flag:
            fused_feature = self.shrink_conv(fused_feature)
        cls_preds, reg_preds, dir_preds = self._run_heads(fused_feature)
        return {'cls_preds': cls_preds, 'reg_preds': reg_preds, 'dir_preds': dir_preds}

    @torch.no_grad()
    def forward(self, data_dict):
        if self.training:
            raise RuntimeError("gencomm_b200 HeterModelBaseline is inference-only: call .eval()")
        affine_matrix = normalize_pairwise_tfm(data_dict['pairwise_t_matrix'], self.H, self.W, self.fake_voxel_size)
        features = {m: self._pad_to_lidar(m, f) for m, f in self._encode(data_dict)}
        heter_feature_2d = self._per_agent(features, data_dict['agent_modality_list'])
        output_dict = self._single_preds(heter_feature_2d)
        output_dict.update(self._detect(heter_feature_2d, data_dict['record_len'], affine_matrix))
        return output_dict
