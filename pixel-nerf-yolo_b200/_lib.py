"""ctypes binding of the C-ABI library (include/pixelnerf_b200.h).

The library is built in-tree (``python -m pixel_nerf_yolo_b200.build`` or ``__graft_entry__.build()``)
as ``pixel-nerf-yolo_b200/csrc/libpixelnerf_b200.so``.  If it is missing, or the device is not sm_100,
every entry point raises: there is no CPU or eager-PyTorch fallback on this path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libpixelnerf_b200.so")

PREC_FP32 = 0
PREC_BF16 = 1
SCENE_MASK_NONNEG_Z = 1
SCENE_RAW_OUTPUT = 2
SCENE_PROJECTED = 4
SCENE_TRAIN_TF32 = 8
SCENE_TRAIN_BF16 = 16
COMBINE_TYPES = {"average": 0, "max": 1}     # pnr_mlp_params.combine_type

# every symbol include/pixelnerf_b200.h declares
EXPORTS = [
    "pnr_version", "pnr_last_error", "pnr_device_supported", "pnr_sample_coarse", "pnr_composite",
    "pnr_sample_fine", "pnr_pack_features", "pnr_gather_encode", "pnr_mlp_pack_bytes", "pnr_mlp_pack",
    "pnr_field_workspace_bytes", "pnr_field_forward", "pnr_last_launch_count", "pnr_gen_rays_yolo", "pnr_yolo_reduce_backward", "pnr_composite_resample",
    "pnr_resnetfc_forward", "pnr_resnetfc_workspace_bytes", "pnr_positional_encoding", "pnr_index_features",
    "pnr_field_tape_bytes", "pnr_field_forward_train", "pnr_field_backward_workspace_bytes", "pnr_field_backward",
    "pnr_composite_backward", "pnr_sample_fine_depth_backward", "pnr_pyramid_pack", "pnr_gen_rays", "pnr_yolo_reduce", "pnr_image_output", "pnr_rgb_loss",
    "pnr_mlp_pack_projected_bytes", "pnr_mlp_pack_projected", "pnr_project_features",
    "pnr_render_workspace_bytes", "pnr_render_forward",
]
# lab equipment (csrc/pnr_lab.h, internal): micro-benchmarks and the tcgen05 self test; not part of the product ABI
LAB_EXPORTS = ["pnr_umma_selftest", "pnr_ingest_bench", "pnr_ingest_bench_tma", "pnr_umma_bench", "pnr_umma2_bench", "pnr_tma_latency_bench", "pnr_dsmem_bench",
               "pnr_lab_gemm_workspace_bytes", "pnr_lab_rowgemm", "pnr_lab_wgrad"]
ABI_VERSION = 3


class Scene(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("poses", C.c_void_p), ("focal", C.c_void_p), ("center", C.c_void_p),
                ("SB", C.c_int32), ("NS", C.c_int32), ("C", C.c_int32), ("Hl", C.c_int32), ("Wl", C.c_int32),
                ("feat_fp32", C.c_int32), ("image_w", C.c_float), ("image_h", C.c_float),
                ("lat_scale_x", C.c_float), ("lat_scale_y", C.c_float), ("flags", C.c_int32)]


class Points(C.Structure):
    _fields_ = [("xyz", C.c_void_p), ("dirs", C.c_void_p), ("rays", C.c_void_p), ("z", C.c_void_p),
                ("mode", C.c_int32), ("P", C.c_int32), ("K", C.c_int32), ("total", C.c_int64),
                ("steps", C.c_void_p), ("noise", C.c_void_p), ("step", C.c_float), ("lindisp", C.c_int32)]


def points_xyz(xyz: "torch.Tensor", dirs: Optional["torch.Tensor"]) -> Points:
    """pnr_points over explicit world points xyz (SB, P, 3) (+ view directions); ``total`` comes from the tensor itself, so
    the library can refuse a scene that was encoded for a different number of objects."""
    pts = Points()
    pts.xyz, pts.dirs, pts.mode, pts.P, pts.K = xyz.data_ptr(), (None if dirs is None else dirs.data_ptr()), 0, xyz.shape[1], 0
    pts.total = xyz.shape[0] * xyz.shape[1]
    return pts


def points_rays(rays: "torch.Tensor", z: "torch.Tensor", sb: int) -> Points:
    """pnr_points over rays (SB*B, 8) x sample depths z (SB*B, K): point (b, k) = o + z[b, k] d."""
    pts = Points()
    Bt, K = z.shape
    assert rays.shape[0] == Bt and Bt % max(sb, 1) == 0
    pts.rays, pts.z, pts.mode, pts.P, pts.K = rays.data_ptr(), z.data_ptr(), 1, (Bt // max(sb, 1)) * K, K
    pts.total = Bt * K
    return pts


class MlpParams(C.Structure):
    _fields_ = [("lin_in_w", C.c_void_p), ("lin_in_b", C.c_void_p), ("lin_out_w", C.c_void_p),
                ("lin_out_b", C.c_void_p), ("fc0_w", C.c_void_p * 8), ("fc0_b", C.c_void_p * 8),
                ("fc1_w", C.c_void_p * 8), ("fc1_b", C.c_void_p * 8), ("linz_w", C.c_void_p * 8),
                ("linz_b", C.c_void_p * 8), ("d_in", C.c_int32), ("d_latent", C.c_int32),
                ("d_hidden", C.c_int32), ("d_out", C.c_int32), ("n_blocks", C.c_int32),
                ("combine_layer", C.c_int32), ("combine_type", C.c_int32)]


class MlpGrads(C.Structure):
    """pnr_mlp_grads: fp32 accumulators laid out like MlpParams (without the dimensions)."""
    _fields_ = [("lin_in_w", C.c_void_p), ("lin_in_b", C.c_void_p), ("lin_out_w", C.c_void_p),
                ("lin_out_b", C.c_void_p), ("fc0_w", C.c_void_p * 8), ("fc0_b", C.c_void_p * 8),
                ("fc1_w", C.c_void_p * 8), ("fc1_b", C.c_void_p * 8), ("linz_w", C.c_void_p * 8),
                ("linz_b", C.c_void_p * 8)]


class RenderArgs(C.Structure):
    """pnr_render_args: NeRFRenderer.forward as one C call."""
    _fields_ = [("scene", C.POINTER(Scene)), ("rays", C.c_void_p), ("B", C.c_int32), ("total_rays", C.c_int64),
                ("scene_fine", C.POINTER(Scene)), ("n_splits", C.c_int32), ("steps", C.c_void_p),
                ("noise_coarse", C.c_void_p), ("noise_u", C.c_void_p), ("noise_jitter", C.c_void_p), ("noise_gauss", C.c_void_p),
                ("mlp_coarse", C.POINTER(MlpParams)), ("packed_coarse", C.c_void_p),
                ("mlp_fine", C.POINTER(MlpParams)), ("packed_fine", C.c_void_p),
                ("n_coarse", C.c_int32), ("n_fine", C.c_int32), ("n_fine_depth", C.c_int32), ("depth_std", C.c_float),
                ("white_bkgd", C.c_int32), ("lindisp", C.c_int32), ("precision", C.c_int32), ("num_freqs", C.c_int32),
                ("freq_factor", C.c_float),
                ("rgb_coarse", C.c_void_p), ("depth_coarse", C.c_void_p), ("weights_coarse", C.c_void_p),
                ("rgb_fine", C.c_void_p), ("depth_fine", C.c_void_p), ("weights_fine", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("field_events", C.c_void_p * 4)]


_lib: Optional[C.CDLL] = None


class NativeLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load (once) and type the library.  Raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). This package has no CPU / eager-PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
    lib.pnr_version.restype = i32
    lib.pnr_last_error.restype = C.c_char_p
    lib.pnr_device_supported.restype = i32
    lib.pnr_last_launch_count.restype = i32
    lib.pnr_sample_coarse.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
    lib.pnr_composite.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.pnr_sample_fine.argtypes = [vp] * 11 + [i32, i32, i32, i32, f32, i32, vp]
    lib.pnr_pack_features.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp]
    lib.pnr_gather_encode.argtypes = [C.POINTER(Scene), C.POINTER(Points), vp, vp, i32, i32, f32, vp]
    lib.pnr_mlp_pack_bytes.argtypes = [C.POINTER(MlpParams)]
    lib.pnr_mlp_pack_bytes.restype = C.c_size_t
    lib.pnr_mlp_pack.argtypes = [C.POINTER(MlpParams), vp, vp]
    lib.pnr_field_workspace_bytes.argtypes = [C.POINTER(Scene), C.POINTER(Points), i32]
    lib.pnr_field_workspace_bytes.restype = C.c_size_t
    lib.pnr_field_forward.argtypes = [C.POINTER(Scene), C.POINTER(Points), C.POINTER(MlpParams), vp, vp, vp,
                                      C.c_size_t, i32, i32, f32, vp]
    lib.pnr_umma_selftest.argtypes = [vp, vp, vp, vp, i32, i32, vp]
    lib.pnr_resnetfc_workspace_bytes.argtypes = [C.POINTER(MlpParams), C.c_longlong]
    lib.pnr_resnetfc_workspace_bytes.restype = C.c_size_t
    lib.pnr_resnetfc_forward.argtypes = [C.POINTER(MlpParams), vp, C.c_longlong, i32, i32, vp, vp, C.c_size_t, vp]
    lib.pnr_positional_encoding.argtypes = [vp, vp, C.c_longlong, i32, i32, f32, i32, vp]
    lib.pnr_index_features.argtypes = [C.POINTER(Scene), vp, i32, i32, vp, vp]
    lib.pnr_ingest_bench.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, i32, vp]
    lib.pnr_ingest_bench_tma.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp]
    lib.pnr_umma_bench.argtypes = [i32, i32, i32, i32, i32, vp, i32, vp]
    lib.pnr_umma2_bench.argtypes = [i32, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.pnr_tma_latency_bench.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp]
    lib.pnr_dsmem_bench.argtypes = [i32, i32, i32, i32, vp, vp]
    lib.pnr_lab_gemm_workspace_bytes.argtypes = [C.c_longlong, i32, i32]
    lib.pnr_lab_gemm_workspace_bytes.restype = C.c_size_t
    lib.pnr_lab_rowgemm.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_longlong, i32, i32, i32, vp, C.c_size_t, vp]
    lib.pnr_lab_wgrad.argtypes = [vp, vp, vp, C.c_longlong, i32, i32, vp, C.c_size_t, vp]
    lib.pnr_field_tape_bytes.argtypes = [C.POINTER(Scene), C.POINTER(Points), C.POINTER(MlpParams)]
    lib.pnr_field_tape_bytes.restype = C.c_size_t
    lib.pnr_field_forward_train.argtypes = [C.POINTER(Scene), C.POINTER(Points), C.POINTER(MlpParams), vp, vp,
                                            C.c_size_t, i32, f32, vp]
    lib.pnr_field_backward_workspace_bytes.argtypes = [C.POINTER(Scene), C.POINTER(Points), C.POINTER(MlpParams)]
    lib.pnr_field_backward_workspace_bytes.restype = C.c_size_t
    lib.pnr_field_backward.argtypes = [C.POINTER(Scene), C.POINTER(Points), C.POINTER(MlpParams), vp, vp, vp,
                                       C.POINTER(MlpGrads), vp, vp, vp, vp, C.c_size_t, i32, f32, vp]
    lib.pnr_composite_backward.argtypes = [vp] * 8 + [i32, i32, i32, vp]
    lib.pnr_sample_fine_depth_backward.argtypes = [vp] * 6 + [i32, i32, i32, f32, vp]
    lib.pnr_pyramid_pack.argtypes = [C.POINTER(vp), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                     i32, i32, vp, i32, vp]
    lib.pnr_mlp_pack_projected_bytes.argtypes = [C.POINTER(MlpParams)]
    lib.pnr_mlp_pack_projected_bytes.restype = C.c_size_t
    lib.pnr_mlp_pack_projected.argtypes = [C.POINTER(MlpParams), vp, vp]
    lib.pnr_project_features.argtypes = [C.POINTER(MlpParams), vp, C.c_longlong, vp, vp, C.c_size_t, vp]
    lib.pnr_render_workspace_bytes.argtypes = [C.POINTER(RenderArgs)]
    lib.pnr_render_workspace_bytes.restype = C.c_size_t
    lib.pnr_render_forward.argtypes = [C.POINTER(RenderArgs), vp]
    lib.pnr_image_output.argtypes = [vp, vp, vp, vp, C.c_longlong, f32, f32, vp]
    lib.pnr_rgb_loss.argtypes = [vp, vp, vp, vp, C.c_longlong, i32, vp]
    lib.pnr_yolo_reduce.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.pnr_yolo_reduce_backward.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.pnr_composite_resample.argtypes = [vp] * 12 + [i32, i32, i32, i32, f32, i32, i32, vp]
    lib.pnr_gen_rays.argtypes = [vp, vp, vp, C.c_longlong, i32, i32, i32, f32, f32, f32, f32, f32, f32, vp]
    lib.pnr_gen_rays_yolo.argtypes = [vp, vp, vp, i32, i32, i32, f32, f32, vp]
    for name in EXPORTS + LAB_EXPORTS:
        getattr(lib, name)          # AttributeError here = header and library disagree
    if lib.pnr_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI version mismatch: library {lib.pnr_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pnr_last_error().decode()
        if rc == -3:
            raise NotImplementedError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on {t.device}: the pixelnerf_b200 path runs on sm_100 GPUs only (no CPU fallback)")


_device_checked = set()


def require_device(device: torch.device) -> None:
    """Fail loudly on anything that is not a B200-class (sm_100) device."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _device_checked:
        return
    with torch.cuda.device(idx):
        if not load().pnr_device_supported():
            raise RuntimeError("pixelnerf_b200: " + load().pnr_last_error().decode())
    _device_checked.add(idx)


def last_launch_count() -> int:
    return load().pnr_last_launch_count()
