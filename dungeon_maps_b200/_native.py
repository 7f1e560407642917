"""ctypes binding of libdungeon_maps_b200.so (the C ABI in include/dungeon_maps_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc when
a toolchain is present, otherwise loading fails loudly; every compute entry
point requires a CUDA device.
"""
import ctypes
import os
from ctypes import POINTER, c_float, c_int32, c_int64, c_size_t, c_void_p

import torch

from . import build as _build

ABI_VERSION = 3


class NativeError(RuntimeError):
  pass


class DmStep(ctypes.Structure):
  _fields_ = [("R", c_float * 9), ("t", c_float * 3), ("kind", c_int32), ("fused", c_int32),
              ("_pad", c_int32 * 2)]


class DmProjCfg(ctypes.Structure):
  _fields_ = [
    ("H", c_int32), ("W", c_int32), ("C", c_int32), ("Mh", c_int32), ("Mw", c_int32),
    ("fx", c_float), ("fy", c_float), ("cx", c_float), ("cy", c_float), ("map_res", c_float),
    ("trunc_depth_min", c_float), ("trunc_depth_max", c_float), ("trunc_height_max", c_float),
    ("has_trunc_depth_min", c_int32), ("has_trunc_depth_max", c_int32), ("has_trunc_height_max", c_int32),
    ("clip_border", c_int32), ("flip_h", c_int32), ("fill_value", c_float), ("want_height", c_int32),
    ("reduction", c_int32), ("fast_steps", c_int32), ("_pad", c_int32 * 3),
  ]


class DmFlowCfg(ctypes.Structure):
  _fields_ = [
    ("H", c_int32), ("W", c_int32), ("channels", c_int32),
    ("fx", c_float), ("fy", c_float), ("cx", c_float), ("cy", c_float),
    ("flip_h", c_int32), ("emit_flow", c_int32), ("_pad", c_int32 * 6),
  ]


class DmFuseSource(ctypes.Structure):
  _fields_ = [
    ("height", c_void_p), ("values", c_void_p), ("mask", c_void_p),
    ("height_bstride", c_int64), ("height_cstride", c_int64),
    ("h", c_int32), ("w", c_int32), ("flip_h", c_int32), ("map_res", c_float),
    ("width_offset", c_void_p), ("height_offset", c_void_p), ("steps", c_void_p), ("plane_box", c_void_p),
  ]


class DmFuseTarget(ctypes.Structure):
  _fields_ = [
    ("Mh", c_int32), ("Mw", c_int32), ("flip_h", c_int32), ("map_res", c_float),
    ("width_offset", c_float), ("height_offset", c_float), ("fill_value", c_float),
    ("reduction", c_int32),
  ]


class DmPoseCfg(ctypes.Structure):
  _fields_ = [("pitch_R", c_float * 9), ("pitch_back_R", c_float * 9), ("cam_height", c_float),
              ("yaw_skew", c_float * 9), ("yaw_skew_sq", c_float * 9), ("fused", c_int32), ("_pad", c_int32 * 2)]


class DmBuilderCfg(ctypes.Structure):
  _fields_ = [
    ("proj", DmProjCfg), ("b", c_int32), ("plot_to_global", c_int32), ("pitch_R", c_float * 9),
    ("cam_height", c_float), ("width_offset", c_float), ("height_offset", c_float),
    ("yaw_skew", c_float * 9), ("yaw_skew_sq", c_float * 9), ("merge_fill_value", c_float),
    ("merge_reduction", c_int32), ("_pad", c_int32 * 2),
  ]


class DmMapRef(ctypes.Structure):
  _fields_ = [("topdown", c_void_p), ("mask", c_void_p), ("h", c_int32), ("w", c_int32),
              ("width_offset", c_float), ("height_offset", c_float), ("box", c_void_p), ("plane_box", c_void_p)]


class DmValueMapRef(ctypes.Structure):
  _fields_ = [("topdown", c_void_p), ("height", c_void_p), ("mask", c_void_p), ("h", c_int32), ("w", c_int32),
              ("width_offset", c_float), ("height_offset", c_float), ("box", c_void_p), ("plane_box", c_void_p)]


class DmMergeShape(ctypes.Structure):
  _fields_ = [("n_valid", c_int64), ("map_height", c_int32), ("map_width", c_int32),
              ("width_offset", c_float), ("height_offset", c_float)]


STEP_WORDS = ctypes.sizeof(DmStep) // 4          # 16
PROJ_SAMPLE_WORDS = 48                           # DmProjSample: 2 steps + 2 offsets + pad
FLOW_SAMPLE_WORDS = 48                           # DmFlowSample: 3 steps
EGO_SAMPLE_WORDS = 20                            # DM_EGO_SAMPLE_WORDS: 1 step + source and window offsets

_SIGNATURES = {
  "dm_abi_version": (ctypes.c_int, []),
  "dm_build_info": (ctypes.c_char_p, []),
  "dm_launch_count": (c_int64, []),
  "dm_sizeof_struct": (c_int32, [c_int32]),
  "dm_release_scratch": (None, []),
  "dm_orth_project_workspace_bytes": (c_size_t, [POINTER(DmProjCfg), c_int32]),
  "dm_orth_project_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(DmProjCfg), c_int32,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
  "dm_orth_project_host_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(DmProjCfg), c_int32,
                                              c_void_p, c_void_p, c_void_p, c_int32]),
  "dm_orth_project_labels_workspace_bytes": (c_size_t, [POINTER(DmProjCfg), c_int32]),
  "dm_orth_project_labels_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(DmProjCfg), c_int32,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
  "dm_orth_project_labels_host_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(DmProjCfg),
                                                     c_int32, c_void_p, c_void_p, c_void_p, c_int32]),
  "dm_upload_params": (ctypes.c_int, [c_void_p, c_size_t, c_void_p, POINTER(c_void_p)]),
  "dm_device_status": (ctypes.c_int, [c_int32]),
  "dm_debug_set_wait_guard": (None, [ctypes.c_uint64, ctypes.c_uint32]),
  "dm_debug_set_host_chunk": (None, [c_int32]),
  "dm_debug_set_tile_rows": (None, [c_int32]),
  "dm_debug_set_dense_shift": (None, [c_int32]),
  "dm_affine_grid_f32": (ctypes.c_int, [c_void_p, c_void_p, POINTER(DmFlowCfg), c_int32, c_void_p, c_void_p]),
  "dm_fuse_bbox_i64": (ctypes.c_int, [POINTER(DmFuseSource), c_int32, c_int32, c_int32, c_float, c_void_p, c_void_p]),
  "dm_fuse_scatter_f32": (ctypes.c_int, [POINTER(DmFuseSource), c_int32, c_int32, c_int32, POINTER(DmFuseTarget),
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
  "dm_fuse_bbox_seeded_i64": (ctypes.c_int, [POINTER(DmFuseSource), c_int32, c_int32, c_int32, c_float, c_void_p,
                                             c_void_p, c_void_p]),
  "dm_fuse_scatter_track_f32": (ctypes.c_int, [POINTER(DmFuseSource), c_int32, c_int32, c_int32, POINTER(DmFuseTarget),
                                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
  "dm_fuse_inplace_f32": (ctypes.c_int, [POINTER(DmFuseSource), c_int32, c_int32, c_int32, POINTER(DmFuseTarget),
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
  "dm_fuse_canvas_init_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, c_void_p]),
  "dm_fuse_clear_envs_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                            POINTER(DmFuseTarget), c_void_p, c_void_p, c_void_p]),
  "dm_pack_proj_samples": (ctypes.c_int, [POINTER(DmPoseCfg), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                          c_int32, c_void_p, POINTER(c_int32)]),
  "dm_pack_flow_samples": (ctypes.c_int, [POINTER(DmPoseCfg), c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
  "dm_pack_ego_samples": (ctypes.c_int, [POINTER(DmPoseCfg), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_int32, c_void_p]),
  "dm_builder_create": (ctypes.c_int, [POINTER(DmBuilderCfg), c_int32, POINTER(c_void_p)]),
  "dm_builder_destroy": (None, [c_void_p]),
  "dm_builder_plot": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     POINTER(DmMapRef), POINTER(DmMergeShape), c_void_p]),
  "dm_builder_plot_prefill": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             POINTER(DmMapRef), POINTER(DmMergeShape), c_void_p, c_void_p, c_int64,
                                             c_void_p]),
  "dm_builder_plot_wait": (ctypes.c_int, [c_void_p, POINTER(DmMergeShape)]),
  "dm_builder_merge": (ctypes.c_int, [c_void_p, POINTER(DmMapRef), c_void_p]),
  "dm_builder_step_fixed": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           POINTER(DmMapRef), c_void_p]),
  "dm_builder_create_values": (ctypes.c_int, [POINTER(DmBuilderCfg), c_int32, c_int32, POINTER(c_void_p)]),
  "dm_builder_plot_values": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_void_p, c_void_p, c_void_p, POINTER(DmValueMapRef), POINTER(DmMergeShape),
                                            c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
  "dm_builder_merge_values": (ctypes.c_int, [c_void_p, POINTER(DmValueMapRef), c_void_p]),
  "dm_builder_step_fixed_values": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p, c_void_p, POINTER(DmValueMapRef), c_void_p]),
  "dm_transform_points_f32": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int64, c_void_p, c_void_p]),
  "dm_image_camera_f32": (ctypes.c_int, [c_void_p, c_int64, c_float, c_float, c_float, c_float, c_int32, c_int32,
                                         c_int32, c_void_p, c_void_p]),
  "dm_depth_to_points_f32": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_float, c_float,
                                            c_float, c_float, c_int32, c_int32, c_float, c_int32, c_float,
                                            c_void_p, c_void_p, c_void_p]),
  "dm_map_quantize_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_float,
                                         c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
  "dm_map_dequantize_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_float,
                                           c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
  "dm_scatter_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int32, c_int32, c_int32,
                                    c_float, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
  "dm_crop_nearest_f32": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                         c_int32, c_float, c_void_p, c_void_p]),
  "dm_crop_nearest_u8": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                        c_void_p, c_void_p]),
  "dm_crop_egocentric_f32": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                            c_float, c_int32, c_void_p, c_int32, c_int32, c_float, c_void_p, c_void_p,
                                            c_void_p, c_void_p]),
  "dm_geodesic_distance_i32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                              c_void_p, c_void_p]),
  "dm_connected_components_i32": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                                 c_void_p, c_void_p]),
  "dm_distance_transform_f32": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
  "dm_score_poses_i32": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_int32, c_void_p,
                                        c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def library_path() -> str:
  return _build.LIB


def lib() -> ctypes.CDLL:
  """Loads (building if needed and possible) the native library.  Never falls back."""
  global _lib
  if _lib is not None:
    return _lib
  path = _build.LIB
  if not os.path.exists(path):
    try:
      _build.build()
    except Exception as e:  # no nvcc on this machine
      raise NativeError(
        f"{path} is missing and could not be built ({e}); run `python -m dungeon_maps_b200.build` "
        "on a machine with nvcc. dungeon_maps_b200 has no CPU fallback.") from e
  handle = ctypes.CDLL(path)
  for name, (res, args) in _SIGNATURES.items():
    fn = getattr(handle, name)  # AttributeError if the .so does not export a declared symbol
    fn.restype = res
    fn.argtypes = args
  if handle.dm_abi_version() != ABI_VERSION:
    raise NativeError(f"ABI mismatch: library {handle.dm_abi_version()} != binding {ABI_VERSION}")
  _lib = handle
  return _lib


def check(rc: int, what: str) -> None:
  if rc == 0:
    return
  if rc > 0:
    raise NativeError(f"{what}: CUDA error {rc}")
  names = {-1: "invalid argument", -2: "workspace too small",
           -3: "a device-side dependency wait timed out in an earlier launch on this device (its outputs are invalid; "
               "the workspace was re-zeroed, the call can be repeated)"}
  raise NativeError(f"{what}: {names.get(rc, rc)}")


def require_cuda(device=None) -> torch.device:
  """The device the kernels will run on.  Raises if there is no CUDA device."""
  if not torch.cuda.is_available():
    raise NativeError("dungeon_maps_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
  if device is None:
    return torch.device("cuda", torch.cuda.current_device())
  device = torch.device(device)
  if device.type != "cuda":
    raise NativeError(f"dungeon_maps_b200 runs on CUDA devices only, got device={device}")
  if device.index is None:
    device = torch.device("cuda", torch.cuda.current_device())
  return device


def ptr(t) -> int:
  return 0 if t is None else t.data_ptr()


def stream_ptr(device: torch.device) -> int:
  """cudaStream_t of torch's current stream on `device` (the raw getter: torch.cuda.current_stream builds a Stream
  object, ~10 us a call, and a MapBuilder step asks a dozen times)."""
  return torch._C._cuda_getCurrentRawStream(device.index if device.index is not None else torch.cuda.current_device())


def device_status(device=None) -> None:
  """Raises NativeError if a projection launch on `device` ran into the dependency-wait guard since the last check
  (include/dungeon_maps_b200.h: dm_device_status).  Synchronise the stream first."""
  dev = require_cuda(device)
  check(lib().dm_device_status(dev.index), "dm_device_status")


def launch_count() -> int:
  return int(lib().dm_launch_count())
