#!/usr/bin/env python
"""distance_transform on config-4 world maps, semantic class planes and random masks: one JSON line per case.

Cases:
  growing / fixed  the world maps of a 32-environment, 100-step MapBuilder walk over synth room scenes
                   (bench.BuilderWorkload geometry, the walk of scripts/time_geodesic.py), on the growing world map and
                   on 2400 x 2400 fixed canvases: the transform of ~obstacle, obstacle = seen and above 0.2 m, i.e. each
                   cell's clearance, the input of the docstring's inflation recipe.
  semantic         the 8 x 16 class planes of the same walk with 16 classes given as class ids: the transform of
                   ~(topdown_map > 0.5), the distance from every cell to the nearest cell of each class.
  random           32 random 2400 x 2400 masks, True with probability 0.99 (1 % of the cells are False).
Arms:
  A  distance_transform without and with return_indices: GPU ms per call from CUDA events around --calls warm calls,
     and the call time (host clock from the call to the end of a device synchronise, median).  Bytes counted from
     shapes (1 B of mask read, 4 B of dist written, 8 B of nearest written) over the event time, next to a device copy
     of the same byte count timed in the same run.
  B  what users do now: a device-to-host copy and scipy.ndimage.distance_transform_edt per plane, cast to float32.
dist must equal B bit for bit and nearest must pass tests/_distance.py's check (asserted on every plane).

usage: python scripts/time_distance.py [--calls 20] [--out results/distance.jsonl]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import ndimage  # noqa: E402

import dungeon_maps_b200 as dmap  # noqa: E402
from scripts.time_components import card, world_map  # noqa: E402
from scripts.time_egocentric import EPISODE, copy_rate  # noqa: E402
from scripts.time_geodesic import world_maps  # noqa: E402
from tests._distance import check_nearest  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def per_pass(mask, calls):
  """GPU ms per call of each pass (edt_rows_kernel, edt_cols_kernel), with indices, from torch.profiler's CUDA
  activities in a run of its own after the timed calls."""
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(calls):
      dmap.distance_transform(mask, return_indices=True)
    torch.cuda.synchronize()
  out = {}
  for ev in prof.key_averages():
    for kernel in ("edt_rows_kernel", "edt_cols_kernel"):
      if kernel in ev.key:
        us = getattr(ev, "device_time_total", None)
        us = ev.cuda_time_total if us is None else us
        out[f"{kernel}_ms"] = round(us / 1e3 / calls, 4)
  return out


def time_case(name, mask, args, extra):
  H, W = mask.shape[-2:]
  planes = mask.numel() // (H * W)
  line = dict(card(), case=name, shape=list(mask.shape), planes=planes, false_cells=int((~mask).sum()), **extra)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  out = {}
  for indices in (False, True):
    res = dmap.distance_transform(mask, return_indices=indices)    # warm the shape
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.calls):
      res = dmap.distance_transform(mask, return_indices=indices)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.calls
    calls = []
    for _ in range(args.calls):
      t0 = time.perf_counter()
      dmap.distance_transform(mask, return_indices=indices)
      torch.cuda.synchronize()
      calls.append((time.perf_counter() - t0) * 1e3)
    nbytes = mask.numel() * (1 + 4 + (8 if indices else 0))
    copy_ms, copy_gbs = copy_rate(nbytes, mask.device)
    key = "indices" if indices else "dist"
    line.update({f"{key}_kernel_ms": round(ms, 4), f"{key}_call_ms_median": round(float(np.median(calls)), 4),
                 f"{key}_bytes": nbytes, f"{key}_larger_than_l2": nbytes > L2_BYTES,
                 f"{key}_GB_per_s": round(nbytes / ms * 1e-6, 1), f"{key}_copy_ms": round(copy_ms, 4),
                 f"{key}_copy_GB_per_s": round(copy_gbs, 1), f"{key}_kernel_over_copy": round(ms / copy_ms, 1)})
    out[key] = res
  line.update(per_pass(mask, args.calls))
  dist, nearest = out["indices"]
  assert torch.equal(out["dist"], dist), f"{name}: dist differs with return_indices"
  t0 = time.perf_counter()
  host = mask.reshape(planes, H, W).cpu().numpy()
  want = np.stack([ndimage.distance_transform_edt(p).astype(np.float32) if not p.all() else
                   np.full(p.shape, np.inf, np.float32) for p in host])
  scipy_ms = (time.perf_counter() - t0) * 1e3
  got = dist.reshape(planes, H, W).cpu().numpy()
  assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"{name}: scipy differs"
  check_nearest(host, got, nearest.reshape(planes, H, W, 2).cpu().numpy())
  line.update(max_dist=float(got[np.isfinite(got)].max()), scipy_planes=planes, scipy_ms=round(scipy_ms, 1),
              scipy_ms_per_plane=round(scipy_ms / planes, 2))
  print(json.dumps(line), flush=True)
  return line


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=20)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,fixed,semantic,random")
  args = ap.parse_args()
  if args.calls < 1:
    ap.error("--calls must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_distance.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  lines = []
  for case in args.cases.split(","):
    if case in ("growing", "fixed"):
      world = world_maps(case == "fixed", dev)
      seen = world.mask[:, 0]
      obstacle = seen & (world.height_map[:, 0] > 0.2)
      lines.append(time_case(f"{case} world map, ~obstacle", (~obstacle).contiguous(), args,
                             extra=dict(steps=EPISODE)))
      del world, seen, obstacle
    elif case == "semantic":
      world = world_map(8, 16, dev)
      lines.append(time_case("semantic world map, ~class planes", ~(world.topdown_map > 0.5), args,
                             extra=dict(steps=EPISODE)))
      del world
    elif case == "random":
      g = torch.Generator(device=dev).manual_seed(0)
      mask = torch.rand((32, 2400, 2400), generator=g, device=dev) < 0.99
      lines.append(time_case("random 2400, 1 % False", mask, args, extra=dict(density=0.99)))
      del mask
    else:
      ap.error(f"unknown case {case}")
    torch.cuda.empty_cache()
  if args.out:
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
      for line in lines:
        f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
  main()
