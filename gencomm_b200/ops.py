"""Tensor-level wrappers over the C ABI: torch supplies device memory and the current stream only.

Every function validates device / dtype / contiguity (the reference's error convention is Python
exceptions, SURVEY.md 8b) and launches asynchronously on ``torch.cuda.current_stream()``.  No
function here synchronises with the host unless its docstring says so.
"""
import ctypes

import numpy as np
import torch

from . import _lib

FUSE_WARP_ONLY, FUSE_MAX, FUSE_ATT = 0, 1, 2
# denoiser arithmetic (include/gencomm_b200.h GC_PREC_*)
PREC_F32, PREC_TC_CONV_IN, PREC_TC_CONV_OUT, PREC_BF16_TC, PREC_TC_MATERIALIZE = 0, 1, 2, 3, 4
PREC_TC_MIDDLE, PREC_TC_ALL, PREC_CLUSTER, PREC_CLUSTER_ALL = 8, 11, 16, 27
MAX_POINTS_PER_PILLAR = 32
MAX_AGENTS_PER_FRAME = 8


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _chk(t, name, dtype, ndim=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (gencomm_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name} must have {ndim} dims, got shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


# --------------------------------------------------------------------------------------------
# geometry / parameter packing (host)
# --------------------------------------------------------------------------------------------
def grid_size(lidar_range, voxel_size):
    """sp_voxel_preprocessor.py:41-43 / heter_encoders.py:25-28: np.round((max-min)/voxel) int64 [nx,ny,nz]."""
    g = (np.array(lidar_range[3:6]) - np.array(lidar_range[0:3])) / np.array(voxel_size)
    return np.round(g).astype(np.int64)


def make_geom(lidar_range, voxel_size, max_voxels, max_points=MAX_POINTS_PER_PILLAR):
    g = grid_size(lidar_range, voxel_size)
    geom = _lib.VoxelGeom()
    for j in range(3):
        geom.range_min[j] = float(lidar_range[j])
        geom.voxel[j] = float(voxel_size[j])
        geom.grid[j] = int(g[j])
    geom.max_points = int(max_points)
    geom.max_voxels = int(max_voxels)
    return geom


def centre_offset(voxel_size, lidar_range):
    """pillar_vfe.py:87-89 (python float64), rounded to fp32 when applied to fp32 tensors."""
    return [voxel_size[j] / 2 + lidar_range[j] for j in range(3)]


def fold_bn(bn_weight, bn_bias, bn_mean, bn_var, eps=1e-3):
    """Eval-mode BatchNorm1d (pillar_vfe.py:25) folded to y = x*scale + shift, in fp32."""
    scale = bn_weight.float() / torch.sqrt(bn_var.float() + eps)
    shift = bn_bias.float() - bn_mean.float() * scale
    return scale, shift


def pack_pfn(weight, bn_weight, bn_bias, bn_mean, bn_var, eps=1e-3):
    """[64,10] Linear weight + BN1d stats -> the [64,16] table of include/gencomm_b200.h (fp32 host math;
    oracle/pillar_ref.c::pack_pfn_row is the same arithmetic)."""
    w = weight.detach().float().cpu()
    if tuple(w.shape) != (64, 10):
        raise ValueError("PillarVFE kernels implement num_filters=[64], 10 input features "
                         "(use_absolute_xyz=True, with_distance=False)")
    scale, shift = fold_bn(bn_weight.detach().cpu(), bn_bias.detach().cpu(), bn_mean.detach().cpu(),
                           bn_var.detach().cpu(), eps)
    t = torch.zeros(64, 16, dtype=torch.float32)
    for j in range(3):
        t[:, j] = ((w[:, j] + w[:, 4 + j]) + w[:, 7 + j]) * scale
        t[:, 4 + j] = w[:, j] * scale
        t[:, 7 + j] = (-w[:, 4 + j]) * scale
    t[:, 3] = w[:, 3] * scale
    t[:, 10] = shift
    t[:, 11] = torch.clamp(shift, min=0.0)
    return t.contiguous()


# --------------------------------------------------------------------------------------------
# (a1) voxelizer
# --------------------------------------------------------------------------------------------
class VoxelWorkspace:
    """Device scratch of gc_voxelize, reusable across calls with the same capacity."""

    def __init__(self, geom, n_agents, total_points, device):
        lib = _lib.load()
        self.geom, self.n_agents, self.total_points = geom, int(n_agents), int(total_points)
        nbytes = lib.gc_voxelize_workspace_bytes(ctypes.byref(geom), self.n_agents, self.total_points)
        if nbytes == 0:
            raise ValueError("bad voxelizer workspace request")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self.n_pillars = torch.empty(self.n_agents, dtype=torch.int32, device=device)


def voxelize(points, point_offsets, ws, max_agent_points=0):
    """points [sumP,4] f32, point_offsets [A+1] i32 (device) -> fills ws, returns ws.n_pillars [A] i32."""
    lib = _lib.load()
    _chk(points, "points", torch.float32, 2)
    _chk(point_offsets, "point_offsets", torch.int32, 1)
    if points.shape[1] != 4:
        raise ValueError("points must be [P,4] (x,y,z,intensity)")
    if point_offsets.numel() != ws.n_agents + 1 or points.shape[0] != ws.total_points:
        raise ValueError("workspace was sized for a different batch")
    _lib.check(lib.gc_voxelize(_ptr(points), _ptr(point_offsets), ws.n_agents, ws.total_points,
                               int(max_agent_points), ctypes.byref(ws.geom), _ptr(ws.buf), _ptr(ws.n_pillars),
                               _stream()), "gc_voxelize")
    return ws.n_pillars


def voxel_gather(points, point_offsets, ws):
    """Reference-shaped (voxel_features [M,32,4], voxel_coords [M,4] i32, voxel_num_points [M] i32).

    Synchronises once to learn sum(M) (the reference API returns exactly-sized arrays)."""
    lib = _lib.load()
    n_pillars = ws.n_pillars
    offs = torch.zeros(ws.n_agents + 1, dtype=torch.int32, device=points.device)
    offs[1:] = torch.cumsum(n_pillars, 0)
    total = int(offs[-1].item())
    voxels = torch.empty(total, 32, 4, dtype=torch.float32, device=points.device)
    coords = torch.empty(total, 4, dtype=torch.int32, device=points.device)
    npts = torch.empty(total, dtype=torch.int32, device=points.device)
    _lib.check(lib.gc_voxel_gather(_ptr(points), _ptr(point_offsets), ws.n_agents, ws.total_points,
                                   ctypes.byref(ws.geom), _ptr(ws.buf), _ptr(offs), total, _ptr(voxels),
                                   _ptr(coords), _ptr(npts), _stream()), "gc_voxel_gather")
    return voxels, coords, npts


# --------------------------------------------------------------------------------------------
# (a3) PillarVFE, (a4) PointPillarScatter, fused front end
# --------------------------------------------------------------------------------------------
def pillar_vfe(voxel_features, voxel_num_points, voxel_coords, pfn, voxel_size, centre_off):
    lib = _lib.load()
    _chk(voxel_features, "voxel_features", torch.float32, 3)
    _chk(voxel_num_points, "voxel_num_points", torch.int32, 1)
    _chk(voxel_coords, "voxel_coords", torch.int32, 2)
    _chk(pfn, "pfn", torch.float32, 2)
    m = voxel_features.shape[0]
    if tuple(voxel_features.shape[1:]) != (32, 4) or tuple(voxel_coords.shape) != (m, 4) \
            or voxel_num_points.shape[0] != m or tuple(pfn.shape) != (64, 16):
        raise ValueError("pillar_vfe: expected voxel_features [M,32,4], coords [M,4], num_points [M], pfn [64,16]")
    out = torch.empty(m, 64, dtype=torch.float32, device=voxel_features.device)
    _lib.check(lib.gc_pillar_vfe(_ptr(voxel_features), _ptr(voxel_num_points), _ptr(voxel_coords), m, _ptr(pfn),
                                 _lib.f3(voxel_size), _lib.f3(centre_off), _ptr(out), _stream()), "gc_pillar_vfe")
    return out


def scatter_canvas(pillar_features, voxel_coords, nx, ny, n_batch, out=None, cell_map=None):
    lib = _lib.load()
    _chk(pillar_features, "pillar_features", torch.float32, 2)
    _chk(voxel_coords, "voxel_coords", torch.int32, 2)
    m, c = pillar_features.shape
    if tuple(voxel_coords.shape) != (m, 4):
        raise ValueError("scatter_canvas: voxel_coords must be [M,4] (b,z,y,x)")
    dev = pillar_features.device
    if out is None:
        out = torch.empty(n_batch, c, ny, nx, dtype=torch.float32, device=dev)
    if cell_map is None:
        cell_map = torch.empty(max(n_batch, 1) * ny * nx, dtype=torch.int32, device=dev)
    _lib.check(lib.gc_scatter_canvas(_ptr(pillar_features), _ptr(voxel_coords), m, c, int(nx), int(ny),
                                     int(n_batch), _ptr(cell_map), _ptr(out), _stream()), "gc_scatter_canvas")
    return out


def plane_bytes(ws):
    """Bytes of one bf16 plane (value or residual) of the canvas of a voxelizer workspace."""
    g = ws.geom
    return max(ws.n_agents * g.grid[1] * g.grid[0] * 64 * 2, 1)


def pillar_canvas_planes(points, point_offsets, ws, pfn, centre_off, out=None, sparse=False):
    """Voxelizer workspace -> BEV canvas as a PlaneFeature (channel-last bf16 value + residual planes, shape [A,64,ny,nx]).
    out = (xh, xl) uint8 buffers of plane_bytes(ws); sparse: the buffers are all-zero, only the occupied cells are written
    (the caller zeroes them again with planes_clear_occupied once the planes have been consumed)."""
    lib = _lib.load()
    _chk(points, "points", torch.float32, 2)
    _chk(point_offsets, "point_offsets", torch.int32, 1)
    _chk(pfn, "pfn", torch.float32, 2)
    g = ws.geom
    if out is None:
        if sparse:
            raise ValueError("pillar_canvas_planes: sparse=True needs the caller's zeroed buffers (out=)")
        xh = torch.empty(plane_bytes(ws), dtype=torch.uint8, device=points.device)
        xl = torch.empty_like(xh)
    else:
        xh, xl = out
        for t in (xh, xl):
            if t.dtype != torch.uint8 or t.numel() != plane_bytes(ws) or t.device != points.device or not t.is_contiguous():
                raise ValueError("pillar_canvas_planes: out must be two contiguous uint8 buffers of plane_bytes(ws)")
    fn = lib.gc_pillar_canvas_planes_sparse if sparse else lib.gc_pillar_canvas_planes
    _lib.check(fn(_ptr(points), _ptr(point_offsets), ws.n_agents, ws.total_points, ctypes.byref(g), _ptr(ws.buf), _ptr(pfn),
                  _lib.f3(centre_off), _ptr(xh), _ptr(xl), _stream()), "gc_pillar_canvas_planes")
    return PlaneFeature(xh, xl, (ws.n_agents, 64, g.grid[1], g.grid[0]))


def planes_clear_occupied(ws, xh, xl):
    """Zeroes the cells pillar_canvas_planes(sparse=True) wrote from this workspace (before its next voxelize)."""
    _lib.check(_lib.load().gc_planes_clear_occupied(ctypes.byref(ws.geom), ws.n_agents, ws.total_points, _ptr(ws.buf), _ptr(xh),
                                                    _ptr(xl), _stream()), "gc_planes_clear_occupied")


def pillar_canvas(points, point_offsets, ws, pfn, centre_off, out=None):
    """Voxelizer workspace -> BEV canvas [A,64,ny,nx] (PFN + scatter fused)."""
    lib = _lib.load()
    _chk(points, "points", torch.float32, 2)
    _chk(point_offsets, "point_offsets", torch.int32, 1)
    _chk(pfn, "pfn", torch.float32, 2)
    g = ws.geom
    if out is None:
        out = torch.empty(ws.n_agents, 64, g.grid[1], g.grid[0], dtype=torch.float32, device=points.device)
    else:
        _chk(out, "out", torch.float32, 4)
        if tuple(out.shape) != (ws.n_agents, 64, g.grid[1], g.grid[0]):
            raise ValueError("pillar_canvas: bad output shape")
    _lib.check(lib.gc_pillar_canvas(_ptr(points), _ptr(point_offsets), ws.n_agents, ws.total_points,
                                    ctypes.byref(g), _ptr(ws.buf), _ptr(pfn), _lib.f3(centre_off), _ptr(out),
                                    _stream()), "gc_pillar_canvas")
    return out


# --------------------------------------------------------------------------------------------
# (a5)-(a9) pose normalisation, warp, fusion
# --------------------------------------------------------------------------------------------
def normalize_pairwise_tfm(pairwise_t_matrix, H, W, discrete_ratio, downsample_rate=1):
    lib = _lib.load()
    _chk(pairwise_t_matrix, "pairwise_t_matrix", torch.float64)
    if tuple(pairwise_t_matrix.shape[-2:]) != (4, 4):
        raise ValueError("pairwise_t_matrix must be [...,4,4]")
    lead = tuple(pairwise_t_matrix.shape[:-2])
    n = int(np.prod(lead)) if lead else 1
    theta = torch.empty(*lead, 2, 3, dtype=torch.float64, device=pairwise_t_matrix.device)
    _lib.check(lib.gc_normalize_pairwise_tfm(_ptr(pairwise_t_matrix), n, float(H), float(W), float(discrete_ratio),
                                             float(downsample_rate), _ptr(theta), _stream()),
               "gc_normalize_pairwise_tfm")
    return theta


def agent_offsets_from_record_len(record_len):
    """record_len [B] (any int dtype, device) -> exclusive prefix [B+1] i32 on the same device, no host sync."""
    off = torch.zeros(record_len.numel() + 1, dtype=torch.int32, device=record_len.device)
    off[1:] = torch.cumsum(record_len.to(torch.int32), 0)
    return off


def warp_fuse(feat, agent_offsets, theta, mode, out=None, max_agents=0):
    """feat [sumN,C,H,W] f32; agent_offsets [B+1] i32; theta [B,L,L,2,3] f64 -> [B,C,H,W] (or [sumN,...]).
    max_agents: host-side upper bound on the agents of any one frame (0 = unknown), lets the library pick the
    kernel specialisation without reading record_len back from the device."""
    lib = _lib.load()
    _chk(feat, "feat", torch.float32, 4)
    _chk(agent_offsets, "agent_offsets", torch.int32, 1)
    _chk(theta, "theta", torch.float64, 5)
    n_frames = agent_offsets.numel() - 1
    total, C, H, W = feat.shape
    B, L = theta.shape[:2]
    if B != n_frames or theta.shape[2] != L or tuple(theta.shape[3:]) != (2, 3):
        raise ValueError("theta must be [B,L,L,2,3] with B == len(record_len)")
    lead = total if mode == FUSE_WARP_ONLY else n_frames
    if out is None:
        out = torch.empty(lead, C, H, W, dtype=torch.float32, device=feat.device)
    else:
        _chk(out, "out", torch.float32, 4)
        if tuple(out.shape) != (lead, C, H, W):
            raise ValueError("warp_fuse: bad output shape")
    _lib.check(lib.gc_warp_fuse(_ptr(feat), _ptr(agent_offsets), n_frames, total, int(max_agents), _ptr(theta), L, C, H, W, int(mode),
                                _ptr(out), _stream()), "gc_warp_fuse")
    return out


# --------------------------------------------------------------------------------------------
# (a10)/(a11) GenComm sampler + DiffusionUNet
# --------------------------------------------------------------------------------------------
def _host_ptr(a):
    if not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]):
        raise TypeError("host blobs must be C-contiguous float32 numpy arrays")
    return a.ctypes.data_as(ctypes.c_void_p)


def _check_blobs(lib, w_host, w_dev, C, T):
    if w_host.size != lib.gc_gencomm_host_weight_floats(T) or w_dev.numel() != lib.gc_gencomm_device_weight_floats(C):
        raise ValueError("packed denoiser weights do not match (C, T)")


def _cluster_ptr(lib, w_cluster, T):
    if w_cluster is None:
        return None
    _chk(w_cluster, "w_cluster", torch.float32, 1)
    if w_cluster.numel() != lib.gc_gencomm_cluster_weight_floats(T):
        raise ValueError("packed cluster-kernel denoiser weights do not match T")
    return _ptr(w_cluster)


def unet_forward(cond, x, t_index, w_host, w_dev, T, workspace=None, precision=0, w_cluster=None):
    """pred = UNet(cat[cond, x], t_index) for all agents; cond [A,2,H,W], x [A,C,H,W] f32."""
    lib = _lib.load()
    _chk(cond, "cond", torch.float32, 4)
    _chk(x, "x", torch.float32, 4)
    _chk(w_dev, "w_dev", torch.float32, 1)
    A, C, H, W = x.shape
    if tuple(cond.shape) != (A, 2, H, W):
        raise ValueError("cond must be [A,2,H,W]")
    _check_blobs(lib, w_host, w_dev, C, T)
    if workspace is None:
        workspace = torch.empty(lib.gc_gencomm_workspace_bytes(A, C, H, W), dtype=torch.uint8, device=x.device)
    pred = torch.empty_like(x)
    _lib.check(lib.gc_unet_forward(_ptr(cond), _ptr(x), A, int(t_index), _host_ptr(w_host), _ptr(w_dev),
                                   _cluster_ptr(lib, w_cluster, T), C, H, W, int(T),
                                   int(precision), _ptr(workspace), _ptr(pred), _stream()), "gc_unet_forward")
    return pred


def unet_trace(cond, x, t_index, w_host, w_dev, T, workspace=None, precision=0, w_cluster=None, pred=None, trace=None):
    """unet_forward that also returns the activations: (pred, [27 NHWC8 tensors]) with tensor 0 = conv_in output and
    tensor 1 + l = the output of middle layer l ([A, H/2, W/2, 8] for l = 4 .. 18, [A, H, W, 8] otherwise).
    pred / trace may be passed in (trace: a flat float32 tensor of gc_unet_trace_floats(A, H, W) elements)."""
    lib = _lib.load()
    _chk(cond, "cond", torch.float32, 4)
    _chk(x, "x", torch.float32, 4)
    _chk(w_dev, "w_dev", torch.float32, 1)
    A, C, H, W = x.shape
    if tuple(cond.shape) != (A, 2, H, W):
        raise ValueError("cond must be [A,2,H,W]")
    _check_blobs(lib, w_host, w_dev, C, T)
    if workspace is None:
        workspace = torch.empty(lib.gc_gencomm_workspace_bytes(A, C, H, W), dtype=torch.uint8, device=x.device)
    n = lib.gc_unet_trace_floats(A, H, W)
    pred = torch.empty_like(x) if pred is None else pred
    trace = torch.empty(n, dtype=torch.float32, device=x.device) if trace is None else trace
    _chk(pred, "pred", torch.float32, 4)
    _chk(trace, "trace", torch.float32, 1)
    if pred.shape != x.shape or trace.numel() != n:
        raise ValueError("unet_trace: pred must be like x and trace must hold gc_unet_trace_floats(A, H, W) floats")
    _lib.check(lib.gc_unet_trace(_ptr(cond), _ptr(x), A, int(t_index), _host_ptr(w_host), _ptr(w_dev),
                                 _cluster_ptr(lib, w_cluster, T), C, H, W, int(T), int(precision), _ptr(workspace),
                                 _ptr(pred), _ptr(trace), _stream()), "gc_unet_trace")
    tensors, off = [], 0
    for k in range(27):
        h, w = (H // 2, W // 2) if 5 <= k <= 19 else (H, W)
        tensors.append(trace[off:off + A * h * w * 8].view(A, h, w, 8))
        off += A * h * w * 8
    return pred, tensors


def gencomm_sample(feat, cond, agent_offsets, noise0, step_noise, w_host, w_dev, schedule, T, workspace=None, out=None,
                   precision=0, w_cluster=None):
    """GenComm eval sampler; feat [sumN,C,H,W], cond [sumN,2,H,W], noise0 like feat, step_noise [>=T-1,sumN,C,H,W]."""
    lib = _lib.load()
    _chk(feat, "feat", torch.float32, 4)
    _chk(cond, "cond", torch.float32, 4)
    _chk(agent_offsets, "agent_offsets", torch.int32, 1)
    _chk(noise0, "noise0", torch.float32, 4)
    _chk(w_dev, "w_dev", torch.float32, 1)
    A, C, H, W = feat.shape
    if tuple(cond.shape) != (A, 2, H, W) or noise0.shape != feat.shape:
        raise ValueError("gencomm_sample: cond must be [A,2,H,W] and noise0 like feat")
    if T > 1:
        _chk(step_noise, "step_noise", torch.float32, 5)
        if step_noise.shape[0] < T - 1 or tuple(step_noise.shape[1:]) != (A, C, H, W):
            raise ValueError("gencomm_sample: step_noise must be [>=T-1, A, C, H, W]")
    _check_blobs(lib, w_host, w_dev, C, T)
    if schedule.shape != (T, 5):
        raise ValueError("schedule must be [T,5]")
    if workspace is None:
        workspace = torch.empty(lib.gc_gencomm_workspace_bytes(A, C, H, W), dtype=torch.uint8, device=feat.device)
    if out is None:
        out = torch.empty_like(feat)
    _lib.check(lib.gc_gencomm_sample(_ptr(feat), _ptr(cond), _ptr(agent_offsets), agent_offsets.numel() - 1, A,
                                     _ptr(noise0), _ptr(step_noise) if T > 1 else None, _host_ptr(w_host), _ptr(w_dev),
                                     _cluster_ptr(lib, w_cluster, T),
                                     _host_ptr(schedule), C, H, W, int(T), int(precision), _ptr(workspace), _ptr(out),
                                     _stream()),
               "gc_gencomm_sample")
    return out


# --------------------------------------------------------------------------------------------
# (8f rank 1) MessageExtractorv2
# --------------------------------------------------------------------------------------------
def me_pack_weights(w_offset, w_dcn):
    """offset1.weight [18,C,3,3], dcn1.weight [64,C,3,3] (device f32) -> packed bf16 B operands (uint8 blob)."""
    lib = _lib.load()
    _chk(w_offset, "offset1.weight", torch.float32, 4)
    _chk(w_dcn, "dcn1.weight", torch.float32, 4)
    C = w_offset.shape[1]
    if tuple(w_offset.shape) != (18, C, 3, 3) or tuple(w_dcn.shape) != (64, C, 3, 3):
        raise ValueError("me_pack_weights: expected offset1.weight [18,C,3,3] and dcn1.weight [64,C,3,3]")
    packed = torch.empty(lib.gc_me_packed_bytes(C), dtype=torch.uint8, device=w_offset.device)
    _lib.check(lib.gc_me_pack_weights(_ptr(w_offset), _ptr(w_dcn), C, _ptr(packed), _stream()), "gc_me_pack_weights")
    return packed


def me_pack_params(sd, prefix="bev_extractor."):
    """The small fp32 parameters in the order include/gencomm_b200.h documents (one device blob)."""
    lib = _lib.load()
    g = lambda k: sd[prefix + k].detach().reshape(-1).float()
    dev = sd[prefix + "dcn1.bias"].device
    z = lambda n: torch.zeros(n, dtype=torch.float32, device=dev)
    blob = torch.cat([g("offset1.bias"), z(14), g("dcn1.bias"), g("attn.1.weight"), g("attn.1.bias"), g("attn.3.weight"),
                      g("attn.3.bias"), g("fuse.0.weight"), g("fuse.0.bias"), g("fuse.2.weight"), g("fuse.2.bias"), z(6)])
    if blob.numel() != lib.gc_me_param_floats():
        raise ValueError("me_pack_params: unexpected parameter shapes")
    return blob.contiguous()


def message_extractor(x, packed, params, workspace=None, out=None):
    """message = MessageExtractorv2(x); x [sumN,C,H,W] f32 (C % 64 == 0, H*W % 128 == 0) -> [sumN,2,H,W]."""
    lib = _lib.load()
    _chk(x, "x", torch.float32, 4)
    _chk(params, "params", torch.float32, 1)
    A, C, H, W = x.shape
    if packed.numel() != lib.gc_me_packed_bytes(C) or params.numel() != lib.gc_me_param_floats():
        raise ValueError("message_extractor: packed weights / params do not match C")
    if workspace is None:
        workspace = torch.empty(lib.gc_me_workspace_bytes(A, C, H, W), dtype=torch.uint8, device=x.device)
    if out is None:
        out = torch.empty(A, 2, H, W, dtype=torch.float32, device=x.device)
    _lib.check(lib.gc_message_extractor(_ptr(x), A, C, H, W, _ptr(packed), _ptr(params), _ptr(workspace), _ptr(out),
                                        _stream()), "gc_message_extractor")
    return out


# --------------------------------------------------------------------------------------------
# (8f rank 1) Enhancer
# --------------------------------------------------------------------------------------------
ENHANCER_PARAM_ORDER = ("block_1.norm1.weight", "block_1.norm1.bias", "block_1.norm2.weight", "block_1.norm2.bias",
                        "block_1.mlp.linear1.0.bias", "block_1.mlp.dwconv.0.weight", "block_1.mlp.dwconv.0.bias",
                        "block_1.mlp.linear2.0.bias", "split_attn.fc1.weight", "split_attn.bn1.weight",
                        "split_attn.bn1.bias", "split_attn.fc2.weight")


def enhancer_pack(sd):
    """state_dict (device tensors) -> (packed bf16x3 B operands, fp32 parameter blob)."""
    lib = _lib.load()
    w_p = sd["block_1.mlp.partial_conv3.weight"].detach().float().contiguous()
    w_1 = sd["block_1.mlp.linear1.0.weight"].detach().float().contiguous()
    w_2 = sd["block_1.mlp.linear2.0.weight"].detach().float().contiguous()
    for t, n in ((w_p, "partial_conv3.weight"), (w_1, "linear1.0.weight"), (w_2, "linear2.0.weight")):
        _chk(t, n, torch.float32)
    C = w_1.shape[1]
    if tuple(w_p.shape) != (C // 4, C // 4, 3, 3) or tuple(w_1.shape) != (4 * C, C) or tuple(w_2.shape) != (C, 2 * C):
        raise ValueError("enhancer_pack: unexpected weight shapes")
    nbytes = lib.gc_enhancer_packed_bytes(C)
    if nbytes == 0:
        raise RuntimeError(f"gc_enhancer: C must be 128 or 256 (got {C})")
    packed = torch.empty(nbytes, dtype=torch.uint8, device=w_1.device)
    _lib.check(lib.gc_enhancer_pack_weights(_ptr(w_p), _ptr(w_1), _ptr(w_2), C, _ptr(packed), _stream()),
               "gc_enhancer_pack_weights")
    params = torch.cat([sd[k].detach().reshape(-1).float() for k in ENHANCER_PARAM_ORDER]).contiguous()
    if params.numel() != lib.gc_enhancer_param_floats(C):
        raise ValueError("enhancer_pack: unexpected parameter shapes")
    return packed, params


def enhancer(x, packed, params, workspace=None, out=None):
    """out = Enhancer(x) for all agents; x [sumN,C,H,W] f32 (C in {128,256}, H*W % 128 == 0)."""
    lib = _lib.load()
    _chk(x, "x", torch.float32, 4)
    _chk(params, "params", torch.float32, 1)
    A, C, H, W = x.shape
    if packed.numel() != lib.gc_enhancer_packed_bytes(C) or params.numel() != lib.gc_enhancer_param_floats(C):
        raise ValueError("enhancer: packed weights / params do not match C")
    if workspace is None:
        workspace = torch.empty(lib.gc_enhancer_workspace_bytes(A, C, H, W), dtype=torch.uint8, device=x.device)
    if out is None:
        out = torch.empty_like(x)
    _lib.check(lib.gc_enhancer(_ptr(x), A, C, H, W, _ptr(packed), _ptr(params), _ptr(workspace), _ptr(out), _stream()),
               "gc_enhancer")
    return out


# --------------------------------------------------------------------------------------------
# (8f rank 2, first slice) DoubleConv (shrink header) and the shared detection heads
# --------------------------------------------------------------------------------------------
def double_conv_pack(w1, b1, w2, b2):
    lib = _lib.load()
    w1, w2 = w1.detach().float().contiguous(), w2.detach().float().contiguous()
    _chk(w1, "double_conv.0.weight", torch.float32, 4)
    _chk(w2, "double_conv.2.weight", torch.float32, 4)
    c_out, c_in = w1.shape[0], w1.shape[1]
    if tuple(w1.shape[2:]) != (3, 3) or tuple(w2.shape) != (c_out, c_out, 3, 3):
        raise NotImplementedError("gencomm_b200 DoubleConv: 3x3 kernels (the shipped shrink headers)")
    packed = torch.empty(max(lib.gc_double_conv_packed_bytes(c_in, c_out), 1), dtype=torch.uint8, device=w1.device)
    _lib.check(lib.gc_double_conv_pack(_ptr(w1), _ptr(w2), c_in, c_out, _ptr(packed), _stream()), "gc_double_conv_pack")
    bias = torch.cat([b1.detach().float().reshape(-1), b2.detach().float().reshape(-1)]).contiguous()
    return packed, bias


def double_conv(x, packed, bias, c_out, stride, workspace=None):
    lib = _lib.load()
    _chk(x, "x", torch.float32, 4)
    A, c_in, H, W = x.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if workspace is None:
        workspace = torch.empty(max(lib.gc_double_conv_workspace_bytes(A, c_in, H, W, stride, c_out), 1), dtype=torch.uint8,
                                device=x.device)
    out = torch.empty(A, c_out, Ho, Wo, dtype=torch.float32, device=x.device)
    _lib.check(lib.gc_double_conv(_ptr(x), A, c_in, H, W, int(stride), int(c_out), _ptr(packed), _ptr(bias), _ptr(workspace),
                                  _ptr(out), _stream()), "gc_double_conv")
    return out


class PlaneFeature:
    """A feature map kept as channel-last bf16 value + residual planes (the tcgen05 convolutions' operand layout) instead of
    NCHW fp32: what BaseBEVBackbone hands to DownsampleConv when both are this package's (``emit_planes``)."""

    def __init__(self, xh, xl, shape):
        self.xh, self.xl, self.shape = xh, xl, tuple(shape)      # shape = (A, C, H, W)
        self.on_consumed = None    # called once by the consumer after its last read of the planes has been enqueued

    def consumed(self):
        cb, self.on_consumed = self.on_consumed, None
        if cb is not None:
            cb()

    @property
    def device(self):
        return self.xh.device


def double_conv_planes(feat, packed, bias, c_out, stride, workspace=None):
    """DoubleConv over a PlaneFeature -> fp32 NCHW [A, c_out, Ho, Wo]."""
    lib = _lib.load()
    A, c_in, H, W = feat.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if workspace is None:
        workspace = torch.empty(max(lib.gc_double_conv_planes_workspace_bytes(A, H, W, stride, c_out), 1), dtype=torch.uint8,
                                device=feat.device)
    out = torch.empty(A, c_out, Ho, Wo, dtype=torch.float32, device=feat.device)
    _lib.check(lib.gc_double_conv_planes(_ptr(feat.xh), _ptr(feat.xl), A, c_in, H, W, int(stride), int(c_out), _ptr(packed),
                                         _ptr(bias), _ptr(workspace), _ptr(out), _stream()), "gc_double_conv_planes")
    return out


def det_heads_pack(weights, biases):
    """weights: 1x1 conv weights [n_i, C, 1, 1] (cls, reg, dir); returns (packed, bias, splits)."""
    lib = _lib.load()
    w = torch.cat([t.detach().float().reshape(t.shape[0], -1) for t in weights]).contiguous()
    _chk(w, "head weights", torch.float32, 2)
    n_out, C = w.shape
    packed = torch.empty(max(lib.gc_det_heads_packed_bytes(C, n_out), 1), dtype=torch.uint8, device=w.device)
    _lib.check(lib.gc_det_heads_pack(_ptr(w), C, n_out, _ptr(packed), _stream()), "gc_det_heads_pack")
    bias = torch.cat([b.detach().float().reshape(-1) for b in biases]).contiguous()
    return packed, bias, [t.shape[0] for t in weights]


def det_heads(x, packed, bias, workspace=None):
    lib = _lib.load()
    _chk(x, "x", torch.float32, 4)
    B, C, H, W = x.shape
    n_out = bias.numel()
    if workspace is None:
        workspace = torch.empty(max(lib.gc_det_heads_workspace_bytes(B, C, H, W), 1), dtype=torch.uint8, device=x.device)
    out = torch.empty(B, n_out, H, W, dtype=torch.float32, device=x.device)
    _lib.check(lib.gc_det_heads(_ptr(x), B, C, H, W, n_out, _ptr(packed), _ptr(bias), _ptr(workspace), _ptr(out), _stream()),
               "gc_det_heads")
    return out


# --------------------------------------------------------------------------------------------
# (8f rank 2) layer primitives over channel-last bf16 planes (BaseBEVBackbone)
# --------------------------------------------------------------------------------------------
def conv_pack(w):
    """w [n_out, c_in, k, k] f32 (k in {1, 3}, BatchNorm folded) -> packed bf16x3 B operand."""
    lib = _lib.load()
    w = w.detach().float().contiguous()
    _chk(w, "conv weight", torch.float32, 4)
    n_out, c_in, k, _ = w.shape
    taps = k * k
    nbytes = lib.gc_conv_packed_bytes(taps, c_in, n_out)
    if nbytes == 0:
        raise NotImplementedError("gencomm_b200 conv layers: 1x1 or 3x3 kernels")
    packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
    _lib.check(lib.gc_conv_pack(_ptr(w), taps, c_in, n_out, _ptr(packed), _stream()), "gc_conv_pack")
    return packed


def to_planes(x):
    """x [A,C,H,W] f32 -> (xh, xl) channel-last bf16 value + residual planes (uint8 blobs)."""
    lib = _lib.load()
    _chk(x, "x", torch.float32, 4)
    A, C, H, W = x.shape
    xh = torch.empty(max(A * H * W * C * 2, 1), dtype=torch.uint8, device=x.device)
    xl = torch.empty_like(xh)
    _lib.check(lib.gc_to_planes(_ptr(x), A, C, H * W, _ptr(xh), _ptr(xl), _stream()), "gc_to_planes")
    return xh, xl


def conv_planes(planes, A, c_in, H_in, W_in, packed, bias, n_out, taps, stride=1, out_nchw=None, out_ch_off=0, up=1,
                up_dy=0, up_dx=0, out_planes=None, out_ch_total=None):
    """ReLU(conv(planes) + bias).  Returns the output planes (xh, xl) when out_nchw is None, else writes into out_nchw
    [A, C_total, Ho*up, Wo*up] at channel offset out_ch_off and phase (up_dy, up_dx).  out_planes = (oh, ol) of
    [A, Ho*up*Wo*up, out_ch_total] bf16 writes the planes into an existing buffer at the same offset / phase."""
    lib = _lib.load()
    xh, xl = planes
    Ho, Wo = ((H_in - 1) // stride + 1, (W_in - 1) // stride + 1) if taps == 9 else (H_in, W_in)
    if out_planes is None and out_nchw is None:    # new planes of exactly this layer's output
        oh = torch.empty(max(A * Ho * Wo * n_out * 2, 1), dtype=torch.uint8, device=xh.device)
        out_planes = (oh, torch.empty_like(oh))
        out_ch_total, out_ch_off, up, up_dy, up_dx = n_out, 0, 1, 0, 0
    if out_planes is not None:
        oh, ol, nchw = _ptr(out_planes[0]), _ptr(out_planes[1]), None
    else:
        _chk(out_nchw, "out", torch.float32, 4)
        oh, ol, nchw, out_ch_total = None, None, _ptr(out_nchw), out_nchw.shape[1]
    _lib.check(lib.gc_conv_planes(_ptr(xh), _ptr(xl), A, c_in, H_in, W_in, stride, taps, n_out, _ptr(packed), _ptr(bias), oh, ol,
                                  nchw, int(out_ch_total), out_ch_off, up, up_dy, up_dx, _stream()), "gc_conv_planes")
    return out_planes, Ho, Wo


# --------------------------------------------------------------------------------------------
# (8f rank 3) decode + rotated NMS
# --------------------------------------------------------------------------------------------
def make_post_params(score_threshold, nms_thresh, dir_offset, num_bins, order, gt_range, top=1000):
    if order not in ("hwl", "lhw"):
        raise ValueError(f"unknown bbx order {order!r}")        # the reference sys.exit()s (voxel_postprocessor.py:119)
    p = _lib.PostParams()
    p.score_threshold, p.nms_thresh, p.dir_offset = float(score_threshold), float(nms_thresh), float(dir_offset)
    p.num_bins, p.order_hwl, p.top = int(num_bins), int(order == "hwl"), int(top)
    for j in range(6):
        p.gt_range[j] = float(gt_range[j])
    return p


def postprocess(cls_preds, reg_preds, dir_preds, anchors, params, tfm=None, workspace=None):
    """cls [B,A,H,W], reg [B,7A,H,W], dir [B,A*bins,H,W] | None, anchors [H,W,A,7] f32, tfm [B,4,4] f32 | None ->
    (boxes [B,top,8,3], scores [B,top], counts [B] i32); rows >= counts[b] are unspecified.  Asynchronous."""
    lib = _lib.load()
    _chk(cls_preds, "cls_preds", torch.float32, 4)
    _chk(reg_preds, "reg_preds", torch.float32, 4)
    _chk(anchors, "anchors", torch.float32, 4)
    B, A, H, W = cls_preds.shape
    if tuple(reg_preds.shape) != (B, 7 * A, H, W) or tuple(anchors.shape) != (H, W, A, 7):
        raise ValueError("postprocess: reg_preds must be [B,7A,H,W] and anchors [H,W,A,7]")
    if dir_preds is not None:
        _chk(dir_preds, "dir_preds", torch.float32, 4)
        if tuple(dir_preds.shape) != (B, A * params.num_bins, H, W):
            raise ValueError("postprocess: dir_preds must be [B,A*num_bins,H,W]")
    if tfm is not None:
        _chk(tfm, "transformation_matrix", torch.float32, 3)
        if tuple(tfm.shape) != (B, 4, 4):
            raise ValueError("postprocess: transformation_matrix must be [B,4,4]")
    dev = cls_preds.device
    if workspace is None:
        workspace = torch.empty(max(lib.gc_postprocess_workspace_bytes(B, A * H * W), 1), dtype=torch.uint8, device=dev)
    boxes = torch.empty(B, params.top, 8, 3, dtype=torch.float32, device=dev)
    scores = torch.empty(B, params.top, dtype=torch.float32, device=dev)
    counts = torch.empty(B, dtype=torch.int32, device=dev)
    _lib.check(lib.gc_postprocess(_ptr(cls_preds), _ptr(reg_preds), _ptr(dir_preds) if dir_preds is not None else None,
                                  _ptr(anchors), _ptr(tfm) if tfm is not None else None, B, A, H, W, ctypes.byref(params),
                                  _ptr(workspace), _ptr(boxes), _ptr(scores), _ptr(counts), _stream()), "gc_postprocess")
    return boxes, scores, counts


# --------------------------------------------------------------------------------------------
# evaluation: greedy detection -> ground-truth matching (eval_utils.caluclate_tp_fp)
# --------------------------------------------------------------------------------------------
EVAL_MAX_BOXES = 1024
EVAL_MAX_THRESHOLDS = 8


def eval_match(det_boxes, det_scores, det_counts, gt_boxes, gt_counts, thresholds, out=None):
    """det_boxes [B,K,8,3] f32, det_scores [B,K] f32, det_counts [B] i32, gt_boxes [B,G,8,3] f32, gt_counts [B] i32 (cuda),
    thresholds: 1..8 IoU thresholds -> (sorted_scores [B,K] f32, tp [B,T,K] u8).  Per frame and threshold the detections
    are sorted by descending score (ties keep input order) and greedily matched, as eval_utils.caluclate_tp_fp does;
    tp[b,t,i] = 1 for a true positive, 0 for a false positive or i >= det_counts[b].  ``out`` = (sorted_scores, tp) to
    write into.  Asynchronous (counts stay on the device; values outside [0, K] / [0, G] are clamped)."""
    lib = _lib.load()
    _chk(det_boxes, "det_boxes", torch.float32, 4)
    _chk(det_scores, "det_scores", torch.float32, 2)
    _chk(det_counts, "det_counts", torch.int32, 1)
    _chk(gt_boxes, "gt_boxes", torch.float32, 4)
    _chk(gt_counts, "gt_counts", torch.int32, 1)
    B, K = det_boxes.shape[:2]
    G = gt_boxes.shape[1]
    if tuple(det_boxes.shape[2:]) != (8, 3) or tuple(det_scores.shape) != (B, K) or tuple(det_counts.shape) != (B,):
        raise ValueError("eval_match: det_boxes must be [B,K,8,3], det_scores [B,K] and det_counts [B]")
    if tuple(gt_boxes.shape) != (B, G, 8, 3) or tuple(gt_counts.shape) != (B,):
        raise ValueError("eval_match: gt_boxes must be [B,G,8,3] and gt_counts [B]")
    if not (1 <= K <= EVAL_MAX_BOXES and 1 <= G <= EVAL_MAX_BOXES):
        raise ValueError(f"eval_match: K and G must be in 1..{EVAL_MAX_BOXES}, got K={K}, G={G}")
    th = np.ascontiguousarray(thresholds, dtype=np.float64).reshape(-1)
    if not 1 <= th.size <= EVAL_MAX_THRESHOLDS:
        raise ValueError(f"eval_match: 1..{EVAL_MAX_THRESHOLDS} thresholds, got {th.size}")
    dev = det_boxes.device
    workspace = torch.empty(lib.gc_eval_workspace_bytes(B, K, G), dtype=torch.uint8, device=dev)
    if out is None:
        out = (torch.empty(B, K, dtype=torch.float32, device=dev), torch.empty(B, th.size, K, dtype=torch.uint8, device=dev))
    sorted_scores, tp = out
    _chk(sorted_scores, "sorted_scores", torch.float32, 2)
    _chk(tp, "tp", torch.uint8, 3)
    if tuple(sorted_scores.shape) != (B, K) or tuple(tp.shape) != (B, th.size, K):
        raise ValueError("eval_match: out must be (sorted_scores [B,K], tp [B,T,K])")
    _lib.check(lib.gc_eval_match(_ptr(det_boxes), _ptr(det_scores), _ptr(det_counts), K, _ptr(gt_boxes), _ptr(gt_counts), G, B,
                                 th.ctypes.data_as(ctypes.c_void_p), th.size, _ptr(workspace), _ptr(sorted_scores), _ptr(tp),
                                 _stream()), "gc_eval_match")
    return sorted_scores, tp


# --------------------------------------------------------------------------------------------
# (8f rank 4) LSS voxel pooling
# --------------------------------------------------------------------------------------------
def lss_voxel_pooling(geom_feats, x, dx, bx, nx, vector=True, deterministic=False):
    """geom_feats [B,N,D,H,W,3] f32, x [B,N,D,H,W,C] f32 (cuda); dx / bx / nx: the three-element tensors of gen_dx_bx
    (host or device) -> [B, nz*C, ny, nx] f32."""
    lib = _lib.load()
    _chk(geom_feats, "geom_feats", torch.float32, 6)
    _chk(x, "x", torch.float32, 6)
    if geom_feats.shape[:5] != x.shape[:5] or geom_feats.shape[5] != 3:
        raise ValueError("lss_voxel_pooling: geom_feats must be [B,N,D,H,W,3] and x [B,N,D,H,W,C]")
    B, C = x.shape[0], x.shape[5]
    dxh = np.ascontiguousarray(torch.as_tensor(dx).detach().cpu().numpy(), dtype=np.float32)
    bxh = np.ascontiguousarray(torch.as_tensor(bx).detach().cpu().numpy(), dtype=np.float32)
    nxh = np.ascontiguousarray(torch.as_tensor(nx).detach().cpu().numpy(), dtype=np.int32)
    out = torch.empty(B, int(nxh[2]) * C, int(nxh[1]), int(nxh[0]), dtype=torch.float32, device=x.device)
    n = x.numel() // C
    nxp = nxh.ctypes.data_as(ctypes.c_void_p)
    if deterministic:   # fixed-point integer reductions: bit-identical run to run (gc_lss_voxel_pooling_det)
        ws = torch.empty(lib.gc_lss_pool_det_workspace_bytes(B, C, nxp), dtype=torch.uint8, device=x.device)
        _lib.check(lib.gc_lss_voxel_pooling_det(_ptr(geom_feats), _ptr(x), n, B, C, dxh.ctypes.data_as(ctypes.c_void_p),
                                                bxh.ctypes.data_as(ctypes.c_void_p), nxp, _ptr(ws), _ptr(out), _stream()),
                   "gc_lss_voxel_pooling_det")
        return out
    ws_bytes = lib.gc_lss_pool_workspace_bytes(B, C, nxp) if vector else 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
    _lib.check(lib.gc_lss_voxel_pooling(_ptr(geom_feats), _ptr(x), n, B, C, dxh.ctypes.data_as(ctypes.c_void_p),
                                        bxh.ctypes.data_as(ctypes.c_void_p), nxp, _ptr(ws) if ws is not None else None,
                                        _ptr(out), _stream()), "gc_lss_voxel_pooling")
    return out
