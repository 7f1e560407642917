#!/usr/bin/env python
"""connected_components on config-4 world maps, semantic class planes, percolation-threshold masks and a spiral: one
JSON line per case.

Cases (8-connectivity):
  growing      the world maps of a 32-environment, 100-step MapBuilder walk over synth room scenes (bench.BuilderWorkload
               geometry, the walk of scripts/time_egocentric.py): the seen mask, the free mask (seen and not above
               0.2 m) and the frontier mask (free cells next to an unseen cell, the docstring's max_pool2d stencil).
  semantic     the 8 x 16 class planes (topdown_map > 0.5) of the same walk with 16 classes given as class ids.
  percolation  32 random 2400 x 2400 masks at the 8-connected site-percolation threshold (density 0.407), where the
               components are largest and most winding.
  spiralN      one N x N one-cell corridor spiral (tests/_geodesic.py): one component that crosses every tile.
Arms:
  A  connected_components, with return_sizes off and on: GPU ms per call from CUDA events around --calls warm calls,
     and the call time (host clock from the call to the end of a device synchronise, median).  Bytes counted from
     shapes (mask read, labels and sizes written) over the event time, next to a device copy of the same byte count
     timed in the same run.
  B  a torch fixed-point min-label propagation on the GPU (every foreground cell takes the smallest index among itself
     and its 8 neighbours), checked for change every 32 iterations, then renumbered in raster order with a cumsum.
  C  what users do now: a device-to-host copy and scipy.ndimage.label per plane.
All three must agree exactly (asserted on the planes each arm ran).  Arm B runs the first 4 planes of the 2400 x 2400
case and skips spirals above 256 x 256 (each iteration moves a label by one cell); every line says how many planes
each arm ran.

usage: python scripts/time_components.py [--calls 20] [--out results/components.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from scipy import ndimage  # noqa: E402

import dungeon_maps_b200 as dmap  # noqa: E402
from scripts.time_egocentric import EPISODE, Walk, copy_rate  # noqa: E402
from scripts.time_reset_envs import make_builder  # noqa: E402
from tests._geodesic import spiral_maze  # noqa: E402

L2_BYTES = 126 * 2 ** 20
CONNECTIVITY = 8


def card():
  name = torch.cuda.get_device_name(0)
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
  except (OSError, subprocess.SubprocessError):
    q = []
  return {"gpu": name, "power_limit": q[0] if len(q) == 2 else "unknown",
          "max_sm_clock": q[1] if len(q) == 2 else "unknown"}


def torch_baseline(mask, check_every=32):
  """(n, H, W) bool -> (labels, counts): min-index propagation over the 8 neighbours until nothing changes."""
  n, H, W = mask.shape
  big = H * W
  idx = torch.arange(H * W, device=mask.device, dtype=torch.int32).view(1, H, W)
  lab = torch.where(mask, idx, big)
  iters = 0
  while True:
    prev = lab
    for _ in range(check_every):
      p = F.pad(lab, (1, 1, 1, 1), value=big)
      best = lab
      for dr in (-1, 0, 1):
        for dc in (-1, 0, 1):
          if dr or dc:
            best = torch.minimum(best, p[:, 1 + dr:1 + dr + H, 1 + dc:1 + dc + W])
      lab = torch.where(mask, best, big)
    iters += check_every
    if torch.equal(lab, prev):
      break
  rank = torch.cumsum((lab == idx).view(n, -1), 1, dtype=torch.int32)    # roots: the cells that kept their index
  out = torch.where(mask, rank.gather(1, lab.view(n, -1).clamp(max=big - 1).long()).view(n, H, W), 0)
  return out, rank[:, -1], iters


def time_case(name, mask, args, torch_planes, extra):
  H, W = mask.shape[-2:]
  planes = mask.numel() // (H * W)
  line = dict(card(), case=name, shape=list(mask.shape), planes=planes, connectivity=CONNECTIVITY,
              foreground_cells=int(mask.sum()), **extra)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  out = {}
  for sizes in (False, True):
    res = dmap.connected_components(mask, CONNECTIVITY, return_sizes=sizes)    # warm the shape
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.calls):
      res = dmap.connected_components(mask, CONNECTIVITY, return_sizes=sizes)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.calls
    calls = []
    for _ in range(args.calls):
      t0 = time.perf_counter()
      dmap.connected_components(mask, CONNECTIVITY, return_sizes=sizes)
      torch.cuda.synchronize()
      calls.append((time.perf_counter() - t0) * 1e3)
    nbytes = mask.numel() * (1 + 4 + (4 if sizes else 0))
    copy_ms, copy_gbs = copy_rate(nbytes, mask.device)
    key = "sizes" if sizes else "labels"
    line.update({f"{key}_kernel_ms": round(ms, 4), f"{key}_call_ms_median": round(float(np.median(calls)), 4),
                 f"{key}_bytes": nbytes, f"{key}_larger_than_l2": nbytes > L2_BYTES,
                 f"{key}_GB_per_s": round(nbytes / ms * 1e-6, 1), f"{key}_copy_ms": round(copy_ms, 4),
                 f"{key}_copy_GB_per_s": round(copy_gbs, 1)})
    out[key] = res
  labels, counts = out["labels"]
  assert torch.equal(out["sizes"][0], labels) and torch.equal(out["sizes"][1], counts)
  flat = mask.reshape(planes, H, W)
  flat_labels, flat_counts = labels.reshape(planes, H, W), counts.reshape(planes)
  line["components_total"] = int(counts.sum())
  if torch_planes:
    k = min(torch_planes, planes)
    m = flat[:k].contiguous()
    torch_baseline(m, 32)                               # warm
    torch.cuda.synchronize()
    e0.record()
    want, want_counts, iters = torch_baseline(m)
    e1.record()
    torch.cuda.synchronize()
    assert torch.equal(want, flat_labels[:k]) and torch.equal(want_counts, flat_counts[:k]), f"{name}: torch differs"
    line.update(torch_planes=k, torch_ms=round(e0.elapsed_time(e1), 3), torch_iterations=iters)
  else:
    line.update(torch_planes=0, torch_ms="not measured")
  structure = np.ones((3, 3), bool)
  t0 = time.perf_counter()
  host = flat.cpu().numpy()
  got = [ndimage.label(p, structure) for p in host]
  scipy_ms = (time.perf_counter() - t0) * 1e3
  assert np.array_equal(np.stack([g[0] for g in got]).astype(np.int32), flat_labels.cpu().numpy()), f"{name}: scipy"
  assert [g[1] for g in got] == flat_counts.cpu().tolist(), f"{name}: scipy counts differ"
  sizes = out["sizes"][2].reshape(planes, H, W).cpu().numpy()
  for p in range(planes):
    per = np.bincount(got[p][0].ravel())
    per[0] = 0
    assert np.array_equal(per[got[p][0]], sizes[p]), f"{name}: sizes differ"
  line.update(scipy_planes=planes, scipy_ms=round(scipy_ms, 1), scipy_ms_per_plane=round(scipy_ms / planes, 2))
  print(json.dumps(line), flush=True)
  return line


def world_map(B, C, dev):
  walk = Walk(B, C, dev)
  builder = make_builder(dev)
  for t in range(EPISODE):
    walk.step(builder, t)
  torch.cuda.synchronize()
  return builder.world_map


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=20)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,semantic,percolation,spiral256,spiral1024")
  args = ap.parse_args()
  if args.calls < 1:
    ap.error("--calls must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_components.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  lines = []
  for case in args.cases.split(","):
    if case == "growing":
      world = world_map(32, 0, dev)
      seen = world.mask[:, 0]
      free = seen & (world.height_map[:, 0] <= 0.2)
      frontier = free & (F.max_pool2d((~seen).float()[:, None], 3, 1, 1)[:, 0] > 0)
      for what, m in (("seen", seen), ("free", free), ("frontier", frontier)):
        lines.append(time_case(f"growing world map, {what}", m.contiguous(), args, torch_planes=32,
                               extra=dict(steps=EPISODE)))
      del world, seen, free, frontier
    elif case == "semantic":
      world = world_map(8, 16, dev)
      lines.append(time_case("semantic world map, class planes", world.topdown_map > 0.5, args, torch_planes=128,
                             extra=dict(steps=EPISODE)))
      del world
    elif case == "percolation":
      g = torch.Generator(device=dev).manual_seed(0)
      mask = torch.rand((32, 2400, 2400), generator=g, device=dev) < 0.407
      lines.append(time_case("percolation 2400", mask, args, torch_planes=4, extra=dict(density=0.407)))
      del mask
    elif case.startswith("spiral"):
      n = int(case[len("spiral"):])
      mask = torch.from_numpy(spiral_maze(n, n))[None].to(dev)
      lines.append(time_case(f"spiral {n}", mask, args, torch_planes=1 if n <= 256 else 0, extra={}))
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
