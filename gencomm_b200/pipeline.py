"""Per-frame collaborative-perception pipeline over the in-scope operators, batched over frames.

    points[F*N*P,4] --voxelize--> workspace --PFN+scatter--> canvas[F*N,64,ny,nx]
    pairwise[F,L,L,4,4] f64 --normalize_pairwise_tfm--> theta[F,L,L,2,3]
    (canvas, theta, record_len) --warp + regroup + Att/Max fusion--> fused[F,64,ny,nx]

This is BASELINE.json config[1] ("PointPillars + AttFusion, 4 agents, 256x256x64 BEV"): the scatter
canvas feeds the fusion directly; the cuDNN backbone/shrink convs that sit between them in the
full detector are out of scope (SURVEY.md section 2.1) and are not part of the measured step.

All buffers are preallocated, every launch is asynchronous on the current stream and nothing
synchronises with the host: the sequence can be enqueued back to back or captured in a CUDA graph.
"""
import numpy as np
import torch

from . import ops
from .modules import PointPillar, SpVoxelPreprocessor

KERNELS_PER_STEP = 7   # cell_assign, pillar_count, pillar_assign, slot_insert, canvas, normalize_tfm, warp_fuse


class FramePipeline:
    def __init__(self, n_frames, n_agents, points_per_agent, lidar_range, voxel_size, max_voxels=70000,
                 fusion="att", max_cav=5, device="cuda", pfn=None):
        self.F, self.N, self.P, self.L = int(n_frames), int(n_agents), int(points_per_agent), int(max_cav)
        self.device = torch.device(device)
        self.lidar_range, self.voxel_size = list(lidar_range), list(voxel_size)
        self.mode = {"att": ops.FUSE_ATT, "max": ops.FUSE_MAX}[fusion]
        self.encoder = PointPillar({"lidar_range": self.lidar_range, "voxel_size": self.voxel_size,
                                    "max_voxels": max_voxels,
                                    "pillar_vfe": {"use_norm": True, "with_distance": False,
                                                   "use_absolute_xyz": True, "num_filters": [64]},
                                    "point_pillar_scatter": {"num_features": 64}})
        if pfn is not None:
            layer = self.encoder.pillar_vfe.pfn_layers[0]
            with torch.no_grad():
                layer.linear.weight.copy_(pfn["weight"]); layer.norm.weight.copy_(pfn["bn_weight"])
                layer.norm.bias.copy_(pfn["bn_bias"]); layer.norm.running_mean.copy_(pfn["bn_mean"])
                layer.norm.running_var.copy_(pfn["bn_var"])
        self.encoder = self.encoder.to(self.device).eval()
        self.pre = SpVoxelPreprocessor(
            {"cav_lidar_range": self.lidar_range,
             "args": {"voxel_size": self.voxel_size, "max_points_per_voxel": 32,
                      "max_voxel_train": max_voxels, "max_voxel_test": max_voxels}}, train=False, device=self.device)
        self.encoder._pre = self.pre
        g = ops.grid_size(self.lidar_range, self.voxel_size)
        self.nx, self.ny = int(g[0]), int(g[1])
        # metric extents, heter_model_baseline.py:87-89 convention (H = y extent, W = x extent, ratio 1)
        self.Hm = self.lidar_range[4] - self.lidar_range[1]
        self.Wm = self.lidar_range[3] - self.lidar_range[0]
        A = self.F * self.N
        self.canvas = torch.empty(A, 64, self.ny, self.nx, dtype=torch.float32, device=self.device)
        self.fused = torch.empty(self.F, 64, self.ny, self.nx, dtype=torch.float32, device=self.device)
        self.agent_offsets = torch.arange(0, A + 1, self.N, dtype=torch.int32, device=self.device)
        self.point_offsets = torch.arange(0, A * self.P + 1, self.P, dtype=torch.int32, device=self.device)

    # algorithmic bytes (SURVEY.md 8d), per step of F frames
    def scatter_bytes(self):
        return self.F * self.N * (16 * self.P + 4 * 64 * self.ny * self.nx)

    def fuse_bytes(self):
        return self.F * (4 * self.N * 64 * self.ny * self.nx + 4 * 64 * self.ny * self.nx + 48 * self.N)

    def encode(self, points, point_offsets=None, events=None):
        """points [F*N*P,4] f32 (device) -> canvas [F*N,64,ny,nx].  events: optional (start, end) pair
        recorded around the canvas writer kernel."""
        off = self.point_offsets if point_offsets is None else point_offsets
        ws = self.pre.voxelize_device(points, off, self.P)
        v = self.encoder.pillar_vfe
        if events:
            events[0].record()
        ops.pillar_canvas(points, off, ws, v.pfn_table(points.device), (v.x_offset, v.y_offset, v.z_offset),
                          out=self.canvas)
        if events:
            events[1].record()
        return self.canvas

    def fuse(self, feat, pairwise, events=None):
        theta = ops.normalize_pairwise_tfm(pairwise, self.Hm, self.Wm, 1.0)
        if events:
            events[0].record()
        ops.warp_fuse(feat, self.agent_offsets, theta, self.mode, out=self.fused, max_agents=self.N)
        if events:
            events[1].record()
        return self.fused

    def step(self, points, pairwise, ev_canvas=None, ev_fuse=None):
        return self.fuse(self.encode(points, events=ev_canvas), pairwise, events=ev_fuse)


def synthetic_step_inputs(step_seed, n_frames, n_agents, points_per_agent, lidar_range, max_cav=5):
    """Host-side (numpy) inputs of one step: points [F*N*P,4] f32 and pairwise [F,L,L,4,4] f64."""
    from . import synth
    clouds, pws = [], []
    half_w = 0.3 * (lidar_range[3] - lidar_range[0])
    half_h = 0.3 * (lidar_range[4] - lidar_range[1])
    for f in range(n_frames):
        frame = step_seed * 1000 + f
        for a in range(n_agents):
            clouds.append(synth.lidar_points(frame, a, points_per_agent, lidar_range=lidar_range))
        pws.append(synth.pairwise_t_matrix(frame, n_agents, max_cav, spread=(half_w, half_h)))
    return np.concatenate(clouds), np.stack(pws)


# ------------------------------------------------------------------------------------------------
# The whole GenComm frame: raw points -> NMS-filtered boxes (BASELINE.json configs[2] / configs[3])
# ------------------------------------------------------------------------------------------------
DETECTOR_STAGES = {"encoder_m1": "pillars", "backbone_m1": "backbone", "shrinker_m1": "shrink",
                   "message_extractor_m1": "message_extractor", "gencomm": "sampler", "enhancer": "enhancer",
                   "fusion_net": "warp_fuse"}


class DetectorPipeline:
    """F collaborative frames per step through ``HeterModelBaselineWGenComm`` (the reference's model call,
    tools/inference_utils.py:141-142) and ``VoxelPostprocessor`` (voxel_postprocessor.py:1084-1244):

        points [F*N*P,4] + pairwise [F,L,L,4,4] f64 -> pillars -> BaseBEVBackbone -> shrink -> MessageExtractorv2 ->
        GenComm sampler (T=3, noise drawn on the device like the reference) -> Enhancer -> warp + Att/Max fusion ->
        heads -> decode + rotated NMS -> boxes [F,1000,8,3], scores [F,1000], counts [F]

    ``shape``: "opv2v_h" (m1_att.yaml: C=128 at 64x128) or "v2xreal" (C=256, z +-15 m; synth.gencomm_v2xreal_args).
    ``detector="baseline"``: ``HeterModelBaseline`` on the same arguments without the GenComm blocks -- the agents share
    their full BEV features and the message extractor, sampler and Enhancer do not run (``precision`` must stay None).
    Everything is asynchronous on the current stream; weights are the seeded synthetic fill of synth.fill_state_dict."""

    def __init__(self, n_frames, n_agents, points_per_agent, shape="opv2v_h", fusion="att", device="cuda", seed=11,
                 score_threshold=0.6, precision=None, detector="gencomm"):
        from . import synth
        from .heter_model_baseline import HeterModelBaseline
        from .heter_model_baseline_w_gencomm_stage1 import HeterModelBaselineWGenComm
        from .postprocess import VoxelPostprocessor
        if detector not in ("gencomm", "baseline"):
            raise ValueError(f"DetectorPipeline: detector {detector!r} -- 'gencomm' or 'baseline'")
        self.F, self.N, self.P = int(n_frames), int(n_agents), int(points_per_agent)
        self.device = torch.device(device)
        self.shape = shape
        self.args = synth.gencomm_v2xreal_args(fusion) if shape == "v2xreal" else synth.gencomm_stage1_args(fusion)
        if detector == "baseline":
            self.args = synth.without_gencomm(self.args)
        self.lidar_range = list(self.args["lidar_range"])
        m = (HeterModelBaseline if detector == "baseline" else HeterModelBaselineWGenComm)(self.args)
        m.load_state_dict(synth.fill_state_dict(m.state_dict(), seed))
        self.model = m.to(self.device).eval()
        if precision is not None:
            self.model.gencomm.precision = precision
        pparams = synth.postprocess_params(score_threshold=score_threshold)
        pparams["gt_range"] = list(self.lidar_range)
        pparams["anchor_args"]["cav_lidar_range"] = list(self.lidar_range)
        self.post = VoxelPostprocessor(pparams, train=False)
        self.anchors = torch.from_numpy(self.post.generate_anchor_box()).float().to(self.device)
        A = self.F * self.N
        self.C = int(self.args["in_head"])
        self.point_offsets = torch.arange(0, A * self.P + 1, self.P, dtype=torch.int32, device=self.device)
        self.record_len = torch.full((self.F,), self.N, dtype=torch.int64, device=self.device)
        self.modalities = ["m1"] * A
        g = ops.grid_size(self.lidar_range, self.args["m1"]["encoder_args"]["voxel_size"])
        self.nx, self.ny = int(g[0]), int(g[1])
        self._marks = None

    # ---- algorithmic work per step (SURVEY.md 8d), the denominators of the per-stage roofline figures ----
    def work(self):
        A, C, H, W = self.F * self.N, self.C, self.ny // 4, self.nx // 4
        b = self.args["m1"]["backbone_args"]
        flops, cin, h, w = 0.0, 64, self.ny, self.nx
        for n, s, f in zip(b["layer_nums"], b["layer_strides"], b["num_filters"]):
            h, w = h // s, w // s
            flops += 2.0 * 9 * cin * f * h * w + n * 2.0 * 9 * f * f * h * w
            cin = f
        h, w = self.ny, self.nx
        for s, f, u, nf in zip(b["layer_strides"], b["num_filters"], b["upsample_strides"], b["num_upsample_filter"]):
            h, w = h // s, w // s
            flops += 2.0 * f * nf * (h * u) * (w * u)
        return {
            "pillars": {"bound": "hbm", "bytes": A * (16 * self.P + 4 * 64 * self.ny * self.nx)},
            "backbone": {"bound": "tensor", "flops": A * flops},
            "warp_fuse": {"bound": "hbm", "bytes": self.F * (4 * self.N * C * H * W + 4 * C * H * W + 48 * self.N)},
            "sampler": {"bound": "hbm", "bytes": A * 3 * (4 * (C + 2) * H * W + 8 * C * H * W),
                        "flops": A * 3 * (486.8e6 if C == 128 else 788.8e6 if C == 256 else 0.0)},
        }

    def enable_stage_timing(self):
        """Forward hooks that record CUDA events around every sub-module the detector has (current stream)."""
        self._marks = []

        def ev():
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            return e
        for name, label in DETECTOR_STAGES.items():
            mod = getattr(self.model, name, None)
            if mod is None:
                continue
            mod.register_forward_pre_hook(lambda _m, _i, label=label: self._mark(label, 0))
            mod.register_forward_hook(lambda _m, _i, _o, label=label: self._mark(label, 1))
        self._ev = ev

    def _mark(self, label, kind):
        if self._marks is not None:      # set to None to stop recording (the hooks stay registered)
            self._marks.append((label, kind, self._ev()))

    def stage_ms(self, n_steps):
        """Mean per-step milliseconds of each stage since the marks were last cleared (call after a synchronize)."""
        per = {}
        for (l0, k0, a), (l1, k1, b) in zip(self._marks[0::2], self._marks[1::2]):
            assert l0 == l1 and k0 == 0 and k1 == 1
            per[l0] = per.get(l0, 0.0) + a.elapsed_time(b) / n_steps
        self._marks.clear()
        return per

    def step(self, points, pairwise, noise=None):
        data = {"inputs_m1": {"points": points, "point_offsets": self.point_offsets, "max_agent_points": self.P},
                "agent_modality_list": self.modalities, "pairwise_t_matrix": pairwise, "record_len": self.record_len}
        if noise is not None:
            data["gencomm_noise"] = noise
        out = self.model(data)
        self._mark("postprocess", 0)
        det = self.post.post_process_batch(out["cls_preds"], out["reg_preds"], out["dir_preds"], self.anchors)
        self._mark("postprocess", 1)
        return det


def synthetic_detector_inputs(step_seed, n_frames, n_agents, points_per_agent, lidar_range, max_cav=5):
    """Host inputs of one detector step: points [F*N*P,4] f32, pairwise [F,L,L,4,4] f64 (agents within ~40 m of the ego so
    that their canvases overlap after the warp, like synth.heter_frames)."""
    from . import synth
    clouds, pws = [], []
    for f in range(n_frames):
        frame = step_seed * 1000 + f
        for a in range(n_agents):
            clouds.append(synth.lidar_points(frame, a, points_per_agent, lidar_range=lidar_range))
        pws.append(synth.pairwise_t_matrix(frame, n_agents, max_cav, spread=(40.0, 15.0)))
    return np.concatenate(clouds), np.stack(pws)
