"""ctypes binding of libgencomm_b200.so (the C ABI of include/gencomm_b200.h).

There is no CPU fallback: if the library is missing or a symbol cannot be resolved the import of
any compute op raises.  PyTorch is used by callers only for device memory and streams; the ABI
itself sees raw pointers.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgencomm_b200.so")

c_int = ctypes.c_int
c_void_p = ctypes.c_void_p
c_double = ctypes.c_double
c_size_t = ctypes.c_size_t


class VoxelGeom(ctypes.Structure):
    """gcVoxelGeom"""
    _fields_ = [("range_min", ctypes.c_float * 3), ("voxel", ctypes.c_float * 3),
                ("grid", ctypes.c_int32 * 3), ("max_points", ctypes.c_int32),
                ("max_voxels", ctypes.c_int32)]


class PostParams(ctypes.Structure):
    """gcPostParams"""
    _fields_ = [("score_threshold", ctypes.c_float), ("nms_thresh", ctypes.c_float), ("dir_offset", ctypes.c_float),
                ("num_bins", ctypes.c_int32), ("order_hwl", ctypes.c_int32), ("top", ctypes.c_int32),
                ("gt_range", ctypes.c_double * 6)]


_F3 = ctypes.c_float * 3
_GEOM_P = ctypes.POINTER(VoxelGeom)

# name -> (restype, argtypes); must list every symbol declared in include/gencomm_b200.h
SIGNATURES = {
    "gc_version": (c_int, []),
    "gc_last_error": (ctypes.c_char_p, []),
    "gc_voxelize_workspace_bytes": (c_size_t, [_GEOM_P, c_int, c_int]),
    "gc_voxelize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, _GEOM_P, c_void_p, c_void_p, c_void_p]),
    "gc_voxel_gather": (c_int, [c_void_p, c_void_p, c_int, c_int, _GEOM_P, c_void_p, c_void_p, c_int,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "gc_pillar_vfe": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, _F3, _F3, c_void_p, c_void_p]),
    "gc_scatter_canvas": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p]),
    "gc_pillar_canvas": (c_int, [c_void_p, c_void_p, c_int, c_int, _GEOM_P, c_void_p, c_void_p, _F3, c_void_p,
                                 c_void_p]),
    "gc_pillar_canvas_planes": (c_int, [c_void_p, c_void_p, c_int, c_int, _GEOM_P, c_void_p, c_void_p, _F3, c_void_p,
                                        c_void_p, c_void_p]),
    "gc_pillar_canvas_planes_sparse": (c_int, [c_void_p, c_void_p, c_int, c_int, _GEOM_P, c_void_p, c_void_p, _F3, c_void_p,
                                               c_void_p, c_void_p]),
    "gc_planes_clear_occupied": (c_int, [_GEOM_P, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gc_warp_fuse": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                             c_void_p, c_void_p]),
    "gc_normalize_pairwise_tfm": (c_int, [c_void_p, c_int, c_double, c_double, c_double, c_double, c_void_p,
                                          c_void_p]),
    "gc_gencomm_host_weight_floats": (c_size_t, [c_int]),
    "gc_gencomm_device_weight_floats": (c_size_t, [c_int]),
    "gc_gencomm_cluster_weight_floats": (c_size_t, [c_int]),
    "gc_gencomm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "gc_gencomm_sample": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gc_unet_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gc_unet_trace_floats": (c_size_t, [c_int, c_int, c_int]),
    "gc_unet_trace": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                              c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gc_me_param_floats": (c_size_t, []),
    "gc_me_packed_bytes": (c_size_t, [c_int]),
    "gc_me_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "gc_me_pack_weights": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gc_message_extractor": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "gc_enhancer_param_floats": (c_size_t, [c_int]),
    "gc_enhancer_packed_bytes": (c_size_t, [c_int]),
    "gc_enhancer_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "gc_enhancer_pack_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gc_enhancer": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gc_double_conv_packed_bytes": (c_size_t, [c_int, c_int]),
    "gc_double_conv_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "gc_double_conv_pack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gc_double_conv": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p]),
    "gc_double_conv_planes_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "gc_double_conv_planes": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "gc_det_heads_packed_bytes": (c_size_t, [c_int, c_int]),
    "gc_det_heads_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "gc_det_heads_pack": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gc_det_heads": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p]),
    "gc_conv_packed_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gc_conv_pack": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gc_to_planes": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gc_conv_planes": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "gc_lss_pool_workspace_bytes": (c_size_t, [c_int, c_int, c_void_p]),
    "gc_lss_voxel_pooling": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
    "gc_lss_pool_det_workspace_bytes": (c_size_t, [c_int, c_int, c_void_p]),
    "gc_lss_voxel_pooling_det": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p]),
    "gc_postprocess_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gc_postprocess": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                               ctypes.POINTER(PostParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gc_eval_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gc_eval_match": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int,
                              c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None


def load():
    """Loads the shared library and binds every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m gencomm_b200.build` "
            "(there is no CPU or PyTorch fallback for the gencomm_b200 kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().gc_last_error().decode(errors="replace")
        kind = "argument error" if rc < 0 else f"CUDA error {rc}"
        raise RuntimeError(f"{what}: {kind}: {msg}")


def f3(vals):
    return _F3(*[float(v) for v in vals])
