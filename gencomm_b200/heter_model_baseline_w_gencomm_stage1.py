"""Drop-in ``HeterModelBaselineWGenComm`` -- the stage-1 GenComm detector, assembled from the B200 operators.

Mirrors ``opencood/models/heter_model_baseline_w_gencomm_stage1.py:31-297``: same constructor argument dict (the
``model.args`` block of ``hypes_yaml/*/GenComm_yamls/gencomm/stage1/*.yaml``), same sub-module names (``encoder_m1``,
``backbone_m1``, ``shrinker_m1``, ``message_extractor_m1``, ``gencomm``, ``enhancer``, ``fusion_net``, ``shrink_conv``,
``cls_head`` / ``reg_head`` / ``dir_head``) so a reference checkpoint loads with ``load_state_dict``, same
``forward(data_dict)`` contract (``tools/inference_utils.py:141-142``):

    data_dict: inputs_m{k} {voxel_features, voxel_coords, voxel_num_points}, agent_modality_list, pairwise_t_matrix
               [B,L,L,4,4] f64, record_len [B]
    returns:   cls_preds, reg_preds, dir_preds, gt_feature, pred_feature, message

and the module file / class name that ``train_utils.create_model`` resolves (``tools/train_utils.py:269-288``; see
``gencomm_b200.create_model``).  Every stage runs a hand-written sm_100a kernel through the C ABI: voxels -> PillarVFE ->
scatter canvas (pillars.cu), BaseBEVBackbone + shrink header (tcgen05 implicit GEMMs), MessageExtractorv2, the GenComm
3-step sampler, Enhancer, warp + Max/Att fusion, detection heads.  Inference only; no CPU path.

Scope: LiDAR ``point_pillar`` modalities and ``fusion_method`` max / att (SURVEY.md section 8a).  Camera modalities
(``lift_splat_shoot``) enter at the encoder boundary: the reference's LSS image encoder (EfficientNet + frustum,
heter_encoders.py:53-300; its voxel pooling is ``gencomm_b200.lss.VoxelPooling``) hands over its BEV feature as
``data_dict['inputs_m{k}']['bev_feature']`` (or is plugged in with ``set_encoder``), and everything behind it -- backbone,
shrink header, message extractor, the CenterCrop zero-padding to the LiDAR extent (:199-213) and the per-agent
re-assembly of the modalities (:215-228) -- runs here.  The other fusion networks and the training-only compressor raise
``NotImplementedError`` at construction.

Extensions (ignored by the reference): ``data_dict['inputs_m{k}']`` may carry raw ``points`` + ``point_offsets`` (see
``modules.PointPillar``); ``data_dict['gencomm_noise'] = (noise0, step_noises)`` injects pre-drawn sampler noise
(parity tests).

The encoder / backbone / shrink header branches, the camera zero-padding, the per-agent re-assembly, the fusion and the
heads are ``HeterModelBaseline``'s (``heter_model_baseline.py``, the same detector without GenComm); this class adds the
message extractors, the sampler and the Enhancer.
"""
import torch

from .enhancer import Enhancer
from .gencomm import GenComm
from .heter_model_baseline import HeterModelBaseline
from .message_extractor import MessageExtractorv2
from .modules import normalize_pairwise_tfm


class HeterModelBaselineWGenComm(HeterModelBaseline):
    GENCOMM_KEY = "gencomm"            # stage 2 reads args['diffcomm'] (…_stage2.py:36)
    MISSING_KEEP = 0.4                 # mask = rand > 0.4 (…_stage1.py:233)
    CROP_MESSAGE = False               # stage 2 pads the camera agents' messages too (…_stage2.py:236); stage 1 does not

    def _add_sampler(self, args):
        self.gencomm = GenComm(args[self.GENCOMM_KEY])
        self.missing_message = args.get('missing_message', False)

    def _add_message_extractor(self, modality_name, args):
        setattr(self, f"message_extractor_{modality_name}", self._make_message_extractor(args))

    def _add_enhancer(self, args):
        if 'enhancer' in args:
            self.enhancer = Enhancer(args['enhancer']['in_ch'], [8, 8], 4)

    @staticmethod
    def _make_message_extractor(args):
        return MessageExtractorv2(args['message_extractor']['in_ch'], args['message_extractor']['out_ch'])

    # hooks the stage-2 class overrides
    def _before_gencomm(self, feature):
        return None

    def _after_gencomm(self, pred, state):
        return pred

    @torch.no_grad()
    def forward(self, data_dict):
        if self.training:
            raise RuntimeError("gencomm_b200 HeterModelBaselineWGenComm is inference-only: call .eval()")
        output_dict = {}
        predraw = 'gencomm_noise' not in data_dict and not self.missing_message
        agent_modality_list = data_dict['agent_modality_list']
        affine_matrix = normalize_pairwise_tfm(data_dict['pairwise_t_matrix'], self.H, self.W, self.fake_voxel_size)
        record_len = data_dict['record_len']

        # predraw: sampler noise of this frame on a side stream, issued between the encoder and the backbone: its generator
        # kernels (HBM writes + ALU) run under the tensor-bound backbone instead of in front of the sampler (after the
        # HBM-bound front end, not beside it; issued after the backbone instead, under the shrink header, it was measured
        # 0.4 % slower: profiles/r02bk)
        features, messages = {}, {}
        for m, feature in self._encode(data_dict, self.gencomm.predraw if predraw else None):
            features[m] = feature
            messages[m] = getattr(self, f"message_extractor_{m}")(feature)

        for m in features:
            features[m] = self._pad_to_lidar(m, features[m])
            if self.CROP_MESSAGE:
                messages[m] = self._pad_to_lidar(m, messages[m])
        heter_feature_2d = self._per_agent(features, agent_modality_list)
        heter_message = self._per_agent(messages, agent_modality_list)

        if self.missing_message:   # robustness experiment: drop message cells of the non-ego agents (…_stage1.py:230-235)
            heter_message = heter_message.clone()
            for i in range(1, heter_message.shape[0]):
                heter_message[i] *= torch.rand(heter_message.shape[1:], device=heter_message.device) > self.MISSING_KEEP
        conditions = heter_message

        output_dict.update(self._single_preds(heter_feature_2d))

        gt_feature = heter_feature_2d
        state = self._before_gencomm(heter_feature_2d)
        gen = self.gencomm(heter_feature_2d, conditions, record_len, noise=data_dict.get('gencomm_noise'))
        pred_feature = gen['pred_feature']
        output_dict.update({'gt_feature': gt_feature, 'pred_feature': pred_feature})
        heter_feature_2d = self._after_gencomm(pred_feature, state)

        if heter_feature_2d.dim() == 3:
            heter_feature_2d = heter_feature_2d.unsqueeze(0)
        if hasattr(self, 'enhancer'):
            heter_feature_2d = self.enhancer(heter_feature_2d, affine_matrix, record_len)
        output_dict.update(self._detect(heter_feature_2d, record_len, affine_matrix))
        output_dict['message'] = conditions
        return output_dict
