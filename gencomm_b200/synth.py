"""Seeded synthetic OPV2V-H-shaped inputs (SURVEY.md section 8d) -- numpy/torch on the host.

There is no dataset on the build or GPU boxes, so every test and bench line uses these generators.
They emit exactly the tensors ``batch['ego']`` carries in the reference
(``intermediate_heter_fusion_dataset.py:596-755``): LiDAR points ``[P,4] f32``, pairwise poses
``[L,L,4,4] f64``, ``record_len [B] i64``, BEV features / messages / pre-drawn sampler noise.
"""
import numpy as np
import torch

OPV2V_H_RANGE = [-102.4, -51.2, -3.0, 102.4, 51.2, 1.0]      # m1_att.yaml:19 -> grid 512x256x1
SQUARE_RANGE = [-51.2, -51.2, -3.0, 51.2, 51.2, 1.0]         # BASELINE config[1] -> grid 256x256x1
VOXEL_SIZE = [0.4, 0.4, 4.0]
BASE_SEED = 20251017


def _rng(frame, agent, salt=0):
    return np.random.default_rng(BASE_SEED + 1000 * int(frame) + int(agent) + 7919 * int(salt))


def lidar_points(frame=0, agent=0, n_points=100_000, lidar_range=OPV2V_H_RANGE, voxel=0.4,
                 uniform=False):
    """LiDAR-like cloud [P,4] f32 (x,y,z,intensity), pre-shuffled (pcd_utils.py:91-95 shuffles).

    64 rings, elevation linspace(-25deg,+2deg), azimuth U[0,2pi), sensor 1.9 m above ground,
    ground-hit range capped at 120 m, 15 % object returns, ~2 % outside the range box and 0.1 %
    snapped exactly onto cell boundaries.  ``uniform=True`` gives the uniform cloud that hits the
    max_voxels cap.
    """
    g = _rng(frame, agent, 1)
    P = int(n_points)
    xmin, ymin, zmin, xmax, ymax, zmax = lidar_range
    if uniform:
        x = g.uniform(xmin, xmax, P)
        y = g.uniform(ymin, ymax, P)
        z = g.uniform(zmin, zmax, P)
    else:
        ring = g.integers(0, 64, P)
        elev = np.deg2rad(np.linspace(-25.0, 2.0, 64))[ring]
        azim = g.uniform(0.0, 2 * np.pi, P)
        down = elev < -1e-3
        r = np.where(down, 1.9 / np.tan(np.where(down, -elev, 1.0)), 120.0)
        r = np.minimum(r, 120.0) * g.uniform(0.97, 1.0, P)
        z = np.where(down & (r < 119.0), -1.9 + g.normal(0, 0.03, P), g.uniform(-1.5, 0.8, P))
        obj = g.random(P) < 0.15
        r = np.where(obj, g.uniform(5.0, 100.0, P), r)
        z = np.where(obj, g.uniform(-1.5, 0.5, P), z)
        x = r * np.cos(azim) + g.normal(0, 0.02, P)
        y = r * np.sin(azim) + g.normal(0, 0.02, P)
    far = g.random(P) < 0.02                      # outside the box -> voxelizer bounds test
    x = np.where(far, x + np.sign(x + 1e-9) * (xmax - xmin), x)
    pts = np.stack([x, y, z, g.random(P)], axis=1).astype(np.float32)
    snap = g.random(P) < 0.001                    # exactly on cell boundaries -> floor() edge
    pts[snap, 0] = (np.round(pts[snap, 0] / voxel) * voxel).astype(np.float32)
    pts[snap, 1] = (np.round(pts[snap, 1] / voxel) * voxel).astype(np.float32)
    g.shuffle(pts, axis=0)
    return np.ascontiguousarray(pts)


def pose_matrix(tx, ty, yaw_deg):
    c, s = np.cos(np.deg2rad(yaw_deg)), np.sin(np.deg2rad(yaw_deg))
    T = np.eye(4)
    T[0, 0], T[0, 1], T[1, 0], T[1, 1] = c, -s, s, c
    T[0, 3], T[1, 3] = tx, ty
    return T


def pairwise_t_matrix(frame=0, n_agents=4, max_cav=5, spread=(60.0, 20.0)):
    """[L,L,4,4] f64, pairwise[i,j] = solve(T_j, T_i) (transformation_utils.py:57-64)."""
    g = _rng(frame, 0, 2)
    Ts = [np.eye(4)]
    for _ in range(1, n_agents):
        Ts.append(pose_matrix(g.uniform(-spread[0], spread[0]), g.uniform(-spread[1], spread[1]),
                              g.uniform(-180.0, 180.0)))
    pw = np.tile(np.eye(4), (max_cav, max_cav, 1, 1))
    for i in range(n_agents):
        for j in range(n_agents):
            if i != j:
                pw[i, j] = np.linalg.solve(Ts[j], Ts[i])
    return pw


def bev_features(frame, n_agents, C, H, W, sparsity=0.0, salt=3):
    g = torch.Generator().manual_seed(BASE_SEED + 1000 * int(frame) + 7919 * salt)
    x = torch.randn(n_agents, C, H, W, generator=g)
    if sparsity > 0:
        keep = torch.rand(n_agents, 1, H, W, generator=g) >= sparsity
        x = x * keep
    return x


def sampler_noise(frame, n_agents, C, H, W, T=3):
    """(noise0, [T step noises]) -- injected into both oracle and kernel (App. A.6 RNG)."""
    g = torch.Generator().manual_seed(BASE_SEED + 1000 * int(frame) + 7919 * 5)
    n0 = torch.randn(n_agents, C, H, W, generator=g)
    steps = [torch.randn(n_agents, C, H, W, generator=g) for _ in range(T)]
    return n0, steps


def pfn_weights(seed=0):
    """PillarVFE parameters: reference default init under manual_seed, BN stats randomised so
    BN is not an identity (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    bound = 1.0 / np.sqrt(10.0)
    w = (torch.rand(64, 10, generator=g) * 2 - 1) * bound          # nn.Linear default: U(-1/sqrt(in), 1/sqrt(in))
    return {
        "weight": w,
        "bn_weight": torch.rand(64, generator=g) * 0.5 + 0.75,
        "bn_bias": torch.randn(64, generator=g) * 0.1,
        "bn_mean": torch.randn(64, generator=g) * 0.1,
        "bn_var": torch.rand(64, generator=g) + 0.5,
    }


def fill_state_dict(state_dict, seed=0):
    """Deterministic, architecture-independent weights for a whole model: every tensor is drawn from a generator seeded
    by (seed, crc32(key)), so the reference model (golden generation) and the drop-in model (tests) get bit-identical
    parameters from their shared ``state_dict`` keys without a multi-MB weight fixture.  Convolution / linear weights
    are scaled to keep activations O(1) through the ReLU stacks; normalisation statistics are non-trivial."""
    import zlib
    out = {}
    for key, ref in state_dict.items():
        g = torch.Generator().manual_seed((int(seed) * 1_000_003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
        shape, leaf = tuple(ref.shape), key.rsplit(".", 1)[-1]
        if not ref.dtype.is_floating_point:
            out[key] = ref.clone()                                        # num_batches_tracked, integer buffers
        elif leaf == "running_var":
            out[key] = torch.rand(shape, generator=g) + 0.5
        elif leaf == "running_mean":
            out[key] = 0.1 * torch.randn(shape, generator=g)
        elif ref.dim() >= 2:
            fan_in = ref[0].numel()
            if "deblocks" in key:                                         # ConvTranspose2d [c_in, c_out, k, k]: one tap per output
                fan_in = ref.shape[0]
            gain = 2.0 if any(s in key for s in ("backbone_", "shrinker_", "shrink_conv")) else 1.0
            if "offset" in key:
                gain = 0.05                                               # deformable offsets stay within a few cells
            out[key] = torch.randn(shape, generator=g) * (gain / max(fan_in, 1)) ** 0.5
        elif leaf == "weight":
            out[key] = 1.0 + 0.2 * torch.randn(shape, generator=g)        # norm scales
        elif leaf == "bias":
            out[key] = 0.1 * torch.randn(shape, generator=g)
        else:                                                             # schedule buffers and other constants stay
            out[key] = ref.clone()
        out[key] = out[key].to(ref.dtype)
    return out


def gencomm_stage1_args(fusion="att"):
    """``model.args`` of hypes_yaml/opv2v/GenComm_yamls/gencomm/stage1/m1_att.yaml:93-170 (LiDAR PointPillars agents,
    OPV2V-H range, C=128 at 64x128) as a fresh dict (the constructors write ``grid_size`` into it)."""
    rng = list(OPV2V_H_RANGE)
    return {
        "ego_modality": "m1", "lidar_range": rng,
        "m1": {"core_method": "point_pillar", "sensor_type": "lidar",
               "encoder_args": {"voxel_size": [0.4, 0.4, 4], "lidar_range": rng,
                                "pillar_vfe": {"use_norm": True, "with_distance": False, "use_absolute_xyz": True,
                                               "num_filters": [64]},
                                "point_pillar_scatter": {"num_features": 64}},
               "backbone_args": {"layer_nums": [3, 5, 8], "layer_strides": [2, 2, 2], "num_filters": [64, 128, 256],
                                 "upsample_strides": [1, 2, 4], "num_upsample_filter": [128, 128, 128]},
               "aligner_args": {"core_method": "identity"},
               "shrink_header": {"kernal_size": [3], "stride": [2], "padding": [1], "dim": [128], "input_dim": 384}},
        "enhancer": {"in_ch": 128}, "message_extractor": {"in_ch": 128, "out_ch": 2},
        "fusion_method": fusion, "att": {"feat_dim": 128}, "in_head": 128, "anchor_number": 2,
        "dir_args": {"dir_offset": 0.7853, "num_bins": 2, "anchor_yaw": [0, 90]}, "gmatch": True,
        "gencomm": {"model": {"embed_dim": 130, "in_channels": 128, "out_ch": 128, "ch": 8, "ch_mult": [1, 1],
                              "num_res_blocks": 2, "attn_resolutions": [16], "dropout": 0.0, "resamp_with_conv": True},
                    "diffusion": {"beta_schedule": "linear", "beta_start": 0.0005, "beta_end": 0.02,
                                  "num_diffusion_timesteps": 3}},
    }


V2XREAL_RANGE = [-102.4, -51.2, -15.0, 102.4, 51.2, 15.0]


def gencomm_v2xreal_args(fusion="att"):
    """V2X-Real-SHAPED ``model.args`` (hypes_yaml/v2xreal/GenComm_yamls/gencomm/stage2/m1m2m3m4_att_infer.yaml:27,51,
    196-326): z range +-15 m with one 30 m voxel, C = 256 at 64 x 128 (shrink header dim 256, enhancer / message extractor /
    AttFusion / heads on 256 channels, denoiser in_channels 256).  All agents use the m1 LiDAR PointPillars branch
    (SURVEY.md App. B.10: m4's identity backbone would give a 256 x 512 map that the reference cannot stack) and the
    single-class head of the OPV2V configs (the yaml's 3-class anchors / multi-class post-processor are outside SURVEY 8)."""
    a = gencomm_stage1_args(fusion)
    rng = list(V2XREAL_RANGE)
    a["lidar_range"] = rng
    a["m1"]["encoder_args"].update({"voxel_size": [0.4, 0.4, 30], "lidar_range": rng})
    a["m1"]["shrink_header"]["dim"] = [256]
    a["enhancer"] = {"in_ch": 256}
    a["message_extractor"] = {"in_ch": 256, "out_ch": 2}
    a["att"] = {"feat_dim": 256}
    a["in_head"] = 256
    a["gencomm"]["model"].update({"embed_dim": 258, "in_channels": 256, "out_ch": 256})
    return a


CAMERA_GRID_CONF = {"xbound": [-51.2, 51.2, 0.4], "ybound": [-51.2, 51.2, 0.4], "zbound": [-10, 10, 20.0],
                    "ddiscr": [2, 50, 48], "mode": "LID"}   # grid_conf_m2 of the OPV2V-H camera yamls: 256 x 256 x 1


def gencomm_stage2_hetero_args(fusion="att"):
    """``model.args`` of hypes_yaml/opv2v/GenComm_yamls/gencomm/stage2/m1m2_att.yaml:150-262 -- LiDAR PointPillars (m1)
    + camera Lift-Splat-Shoot (m2) agents.  m2: the LSS encoder emits a 128-channel BEV feature on the 256 x 256 camera
    grid (+-51.2 m), one backbone level + shrink header take it to 128 x 64 x 64, and the model zero-pads it to the LiDAR
    extent 64 x 128 (crop ratio W = 102.4 / 51.2).  The sampler block sits under ``diffcomm`` (what the class reads)."""
    a = gencomm_stage1_args(fusion)
    a["diffcomm"] = a.pop("gencomm")
    a["m2"] = {"core_method": "lift_splat_shoot", "sensor_type": "camera",
               "encoder_args": {"anchor_number": 2, "grid_conf": dict(CAMERA_GRID_CONF), "img_downsample": 8,
                                "img_features": 128, "use_depth_gt": False, "depth_supervision": False,
                                "camera_encoder": "EfficientNet"},
               "camera_mask_args": {"cav_lidar_range": list(OPV2V_H_RANGE), "grid_conf": dict(CAMERA_GRID_CONF)},
               "backbone_args": {"layer_nums": [3], "layer_strides": [2], "num_filters": [64], "upsample_strides": [1],
                                 "num_upsample_filter": [128], "inplanes": 128},
               "aligner_args": {"core_method": "identity"},
               "shrink_header": {"kernal_size": [3], "stride": [2], "padding": [1], "dim": [128], "input_dim": 128}}
    return a


def without_gencomm(args):
    """``model.args`` of a GenComm detector minus its GenComm blocks (sampler, Enhancer, message extractor): the arguments
    of ``HeterModelBaseline``, the same detector sending full BEV features."""
    return {k: v for k, v in args.items() if k not in ("gencomm", "diffcomm", "enhancer", "message_extractor")}


def heter_baseline_args(fusion="att"):
    """``HeterModelBaseline`` arguments of the LiDAR PointPillars agents of ``gencomm_stage1_args`` (OPV2V-H range, C=128
    at 64x128) -- BASELINE.json configs 1-2."""
    return without_gencomm(gencomm_stage1_args(fusion))


def heter_baseline_hetero_args(fusion="att"):
    """``HeterModelBaseline`` arguments of the LiDAR (m1) + camera (m2) agents of ``gencomm_stage2_hetero_args``."""
    return without_gencomm(gencomm_stage2_hetero_args(fusion))


def heter_frames(seed, record_len, n_points=30_000, max_cav=5):
    """Host inputs of a batch of collaborative frames for the full detector: per-agent clouds (list of [P,4] f32) and
    ``pairwise_t_matrix`` [B,L,L,4,4] f64; agents stay within ~40 m so their canvases overlap after the warp."""
    clouds, pws = [], []
    for f, n in enumerate(record_len):
        for a in range(int(n)):
            clouds.append(lidar_points(seed + f, a, n_points))
        pws.append(pairwise_t_matrix(seed + f, int(n), max_cav, spread=(40.0, 15.0)))
    return clouds, np.stack(pws)


def postprocess_params(score_threshold=0.2, nms_thresh=0.15):
    """``postprocess`` block of m1_att.yaml:66-89 with the fields yaml_utils.load_point_pillar_params adds (:71-80)."""
    rng = list(OPV2V_H_RANGE)
    return {"core_method": "VoxelPostprocessor", "gt_range": rng, "order": "hwl", "max_num": 150, "nms_thresh": nms_thresh,
            "anchor_args": {"cav_lidar_range": rng, "l": 3.9, "w": 1.6, "h": 1.56, "r": [0, 90], "feature_stride": 4,
                            "num": 2, "vw": 0.4, "vh": 0.4, "W": 512, "H": 256},
            "target_args": {"pos_threshold": 0.6, "neg_threshold": 0.45, "score_threshold": score_threshold},
            "dir_args": {"dir_offset": 0.7853, "num_bins": 2, "anchor_yaw": [0, 90]}}


def head_outputs(seed, H=64, W=128, A=2, bins=2, bias=-3.0, smooth=5):
    """Synthetic detector head maps of one frame: cls [1,A,H,W] (spatially smooth so that positives cluster and the NMS
    has overlapping boxes to suppress; ``bias`` sets the candidate count), reg [1,7A,H,W], dir [1,A*bins,H,W]."""
    g = torch.Generator().manual_seed(int(seed))
    raw = torch.randn(1, A, H + smooth - 1, W + smooth - 1, generator=g)
    cls = torch.nn.functional.avg_pool2d(raw, smooth, stride=1) * (1.2 * smooth) + bias
    reg = 0.3 * torch.randn(1, 7 * A, H, W, generator=g)
    dr = torch.randn(1, A * bins, H, W, generator=g)
    return cls.contiguous(), reg, dr


LSS_GRID_CONF = {"xbound": [-51.2, 51.2, 0.4], "ybound": [-51.2, 51.2, 0.4], "zbound": [-10, 10, 20.0],
                 "ddiscr": [2, 50, 48]}     # the camera grid of the OPV2V-H LSS agents (m2 yaml blocks): 256 x 256 x 1


def lss_frustum(seed, B=2, N=2, D=12, H=8, W=11, C=16, grid_conf=None, coarse_frac=0.5):
    """Synthetic frustum: geom_feats [B,N,D,H,W,3] (ego-frame xyz; ~10 % outside the grid, some within one cell below the
    lower bound, where the reference's truncation keeps them) and features x [B,N,D,H,W,C].  ``coarse_frac`` of the
    points are snapped onto a 3 m lattice (many points per cell: exercises the accumulation)."""
    conf = grid_conf or LSS_GRID_CONF
    g = torch.Generator().manual_seed(int(seed))
    shape = (B, N, D, H, W)
    xs = (torch.rand(shape, generator=g) * 1.12 - 0.06) * (conf["xbound"][1] - conf["xbound"][0]) + conf["xbound"][0]
    ys = (torch.rand(shape, generator=g) * 1.12 - 0.06) * (conf["ybound"][1] - conf["ybound"][0]) + conf["ybound"][0]
    zs = (torch.rand(shape, generator=g) * 1.2 - 0.1) * (conf["zbound"][1] - conf["zbound"][0]) + conf["zbound"][0]
    # camera rays hit the same cells many times: quantise half of the points onto a coarse lattice
    coarse = torch.rand(shape, generator=g) < coarse_frac
    xs = torch.where(coarse, torch.round(xs / 3.0) * 3.0 + 0.1, xs)
    ys = torch.where(coarse, torch.round(ys / 3.0) * 3.0 + 0.1, ys)
    geom = torch.stack([xs, ys, zs], dim=-1).float()
    x = torch.randn(*shape, C, generator=g)
    return geom, x


_CORNER_TEMPLATE = np.array([[1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, -1],
                             [1, -1, 1], [1, 1, 1], [-1, 1, 1], [-1, -1, 1]], dtype=np.float64) / 2


def box_corners(boxes):
    """[N,7] (x, y, z, l, w, h, yaw) -> [N,8,3] f32 corners in the order of box_utils.boxes_to_corners_3d (order 'lhw',
    utils/box_utils.py:152-203): template (+-l/2, +-w/2, +-h/2), rotation by yaw about z, then the centre."""
    b = np.asarray(boxes, dtype=np.float64).reshape(-1, 7)
    c = b[:, None, 3:6] * _CORNER_TEMPLATE[None]
    co, si = np.cos(b[:, 6])[:, None], np.sin(b[:, 6])[:, None]
    x = c[..., 0] * co - c[..., 1] * si + b[:, None, 0]
    y = c[..., 0] * si + c[..., 1] * co + b[:, None, 1]
    return np.stack([x, y, c[..., 2] + b[:, None, 2]], axis=-1).astype(np.float32)


def _cars(g, n):
    """n car-sized boxes [n,7] (l 3.5-5, w 1.6-2.1, h 1.4-1.8 m, any yaw) with all corners inside the OPV2V-H gt_range."""
    xmin, ymin, _, xmax, ymax, _ = OPV2V_H_RANGE
    return np.stack([g.uniform(xmin + 3.5, xmax - 3.5, n), g.uniform(ymin + 3.5, ymax - 3.5, n), g.uniform(-1.9, -0.9, n),
                     g.uniform(3.5, 5.0, n), g.uniform(1.6, 2.1, n), g.uniform(1.4, 1.8, n),
                     g.uniform(-np.pi, np.pi, n)], axis=1)


def _jitter(g, boxes, pos, size, yaw):
    out = boxes.copy()
    out[:, 0:2] += g.normal(0.0, pos, (len(boxes), 2))
    out[:, 3:5] *= 1.0 + g.normal(0.0, size, (len(boxes), 2))
    out[:, 6] += g.normal(0.0, yaw, len(boxes))
    return out


def eval_frames(seed, n_frames, k_max=1000, g_max=200, n_gt=(20, 200), no_det=(), no_gt=(), full=(), score_step=None):
    """Padded detections and ground truths of ``n_frames`` frames for the evaluation matching (eval_utils.caluclate_tp_fp):

        det_boxes [B,k_max,8,3] f32, det_scores [B,k_max] f32, det_counts [B] i32,
        gt_boxes [B,g_max,8,3] f32, gt_counts [B] i32       (torch, host; rows beyond a count are zero)

    Ground truths: n_gt[0]..n_gt[1] car-sized boxes (at most g_max) with random yaw inside the OPV2V-H range.  Detections,
    in random order: a jittered copy of ~80 % of the ground truths, a second, looser copy of ~30 % of those (duplicates,
    so the greedy order matters) and free false positives; scores U(0.2, 1), rounded to multiples of ``score_step`` if
    given (many equal scores).  Frames listed in ``no_det`` have no detection, in ``no_gt`` no ground truth, and in
    ``full`` exactly k_max detections."""
    B = int(n_frames)
    det = np.zeros((B, k_max, 8, 3), np.float32)
    scores = np.zeros((B, k_max), np.float32)
    gts = np.zeros((B, g_max, 8, 3), np.float32)
    det_counts = np.zeros(B, np.int32)
    gt_counts = np.zeros(B, np.int32)
    for f in range(B):
        g = np.random.default_rng(BASE_SEED + 1000 * int(seed) + 7919 * 11 + f)
        n_g = 0 if f in no_gt else min(int(g.integers(n_gt[0], n_gt[1] + 1)), g_max)
        gt = _cars(g, n_g)
        hit = gt[g.random(n_g) < 0.8]
        dup = hit[g.random(len(hit)) < 0.3]
        parts = [_jitter(g, hit, 0.25, 0.06, 0.08), _jitter(g, dup, 0.6, 0.1, 0.2),
                 _cars(g, int(g.integers(2, 10 + n_g // 5)))]
        d = np.concatenate(parts)
        if f in full and len(d) < k_max:
            d = np.concatenate([d, _cars(g, k_max - len(d))])
        d = d[g.permutation(len(d))][:k_max]
        if f in no_det:
            d = d[:0]
        s = g.uniform(0.2, 1.0, len(d))
        if score_step:
            s = np.round(s / score_step) * score_step
        gts[f, :n_g] = box_corners(gt)
        det[f, :len(d)] = box_corners(d)
        scores[f, :len(d)] = s.astype(np.float32)
        det_counts[f], gt_counts[f] = len(d), n_g
    return {"det_boxes": torch.from_numpy(det), "det_scores": torch.from_numpy(scores),
            "det_counts": torch.from_numpy(det_counts), "gt_boxes": torch.from_numpy(gts),
            "gt_counts": torch.from_numpy(gt_counts)}
