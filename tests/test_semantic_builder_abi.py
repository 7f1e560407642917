"""The semantic MapBuilder step's C ABI without a device: the DmValueMapRef mirror against the compiled struct, and the
argument checks of dm_builder_create_values, which refuse bad configurations before any CUDA call."""
import ctypes

import pytest

from dungeon_maps_b200 import _native as nat


def test_value_map_ref_layout():
  lib = nat.lib()
  R = nat.DmValueMapRef
  assert ctypes.sizeof(R) == lib.dm_sizeof_struct(11) == 3 * 8 + 4 * 4 + 2 * 8
  assert [R.topdown.offset, R.height.offset, R.mask.offset] == [0, 8, 16]
  assert [R.h.offset, R.w.offset, R.width_offset.offset, R.height_offset.offset] == [24, 28, 32, 36]
  assert [R.box.offset, R.plane_box.offset] == [40, 48]
  assert lib.dm_sizeof_struct(12) == -1


def _cfg(C, reduction=0, merge_reduction=0):
  cfg = nat.DmBuilderCfg()
  p = cfg.proj
  p.H, p.W, p.C, p.Mh, p.Mw = 48, 64, C, 40, 40
  p.map_res, p.reduction = 0.05, reduction
  cfg.b, cfg.plot_to_global = 2, 0
  cfg.merge_reduction = merge_reduction
  return cfg


@pytest.mark.parametrize("case", ["C=0 values", "C=0 labels", "C=64 labels", "C=-1 values", "sum", "merge prod",
                                  "b=0", "Mh=0"])
def test_create_values_refuses_bad_arguments(case):
  lib = nat.lib()
  labels = 1 if "labels" in case else 0
  cfg = {"C=0 values": _cfg(0), "C=0 labels": _cfg(0), "C=64 labels": _cfg(64), "C=-1 values": _cfg(-1),
         "sum": _cfg(4, reduction=2), "merge prod": _cfg(4, merge_reduction=4), "b=0": _cfg(4), "Mh=0": _cfg(4)}[case]
  if case == "b=0":
    cfg.b = 0
  if case == "Mh=0":
    cfg.proj.Mh = 0
  handle = ctypes.c_void_p()
  assert lib.dm_builder_create_values(cfg, labels, 0, ctypes.byref(handle)) == -1
  assert not handle.value


def test_create_values_refuses_null_pointers():
  lib = nat.lib()
  handle = ctypes.c_void_p()
  assert lib.dm_builder_create_values(None, 0, 0, ctypes.byref(handle)) == -1
  assert lib.dm_builder_create_values(_cfg(4), 0, 0, None) == -1
  # the height-map entry keeps refusing value channels, and the step entries of both kinds refuse a missing handle
  assert lib.dm_builder_create(_cfg(4), 0, ctypes.byref(handle)) == -1
  assert lib.dm_builder_merge_values(None, None, None) == -1
  assert lib.dm_builder_plot_values(None, *([None] * 14), 0, None) == -1
  assert lib.dm_builder_step_fixed_values(None, *([None] * 11)) == -1
  assert lib.dm_builder_plot(None, *([None] * 9)) == -1
  assert lib.dm_builder_plot_prefill(None, *([None] * 10), 0, None) == -1
  assert lib.dm_builder_plot_wait(None, None) == -1
  assert lib.dm_builder_merge(None, None, None) == -1
  assert lib.dm_builder_step_fixed(None, *([None] * 8)) == -1
