#!/usr/bin/env python
"""score_poses on config-4 world maps: one JSON line per case and lattice.

The walk is the one the other time_*.py scripts share (bench.BuilderWorkload geometry over synth room scenes, 480x640
depth -> 400x400 local maps at 3 cm, 100 steps): steps 0..98 build the world map at their true poses, and the local map
of step 99, plotted in its camera frame and not merged, is the window (width_offset=200, height_offset=0).  Cases:
  obstacle          32 environments, growing world map, planes = world obstacle cells (seen and above 0.2 m), window =
                    the local obstacle cells;
  obstacle+free     the same, planes = world obstacle and world free cells (2 planes, one shared window);
  seen              the same walk, planes = world seen cells, window = every seen cell of the local map: a dense
                    window, for the kernel's rate (the obstacle windows of this walk are nearly empty);
  fixed             the same two planes on 2400 x 2400 fixed canvases;
  semantic          8 environments with 16 classes given as class ids: planes = world class planes (> 0.5), one window
                    per plane = the local class planes.
Lattices around step 99's true pose: 11 x 11 x 11 (+-5 cells, +-5 degrees, 1331 candidates) and 5 x 5 x 5.
Per case and lattice:
  A  score_poses: kernel ms from CUDA events around --calls warm calls, call ms (host clock to a device synchronise,
     median), host ms packing and uploading the candidates (prm.ego_samples + upload, median), per-pass ms from
     torch.profiler in a run of its own, cell-candidate evaluations (True window cells x candidates, per window plane)
     per second of kernel time;
  B  the crop_egocentric_map loop over the candidates, ANDed with the window and summed on the device: ms for all
     candidates; equal to A bit for bit (asserted);
  C  a device-to-host copy and the numpy oracle (tests/_match.py) on a fixed subset of --oracle candidates: measured ms
     per candidate (copy excluded, reported apart); equal to A on that subset (asserted).
For the obstacle+free and fixed cases, also the docstring's recipe: the odometry pose is step 99's true pose plus
(3 cells, -2 cells, 3 degrees), the 1331-candidate lattice is centred on it, the score is s[:, 0] - s[:, 1], and the
line reports how many environments the argmax puts within one lattice step of the true pose, and score margins.

usage: python scripts/time_score_poses.py [--calls 20] [--oracle 8] [--out results/score_poses.jsonl]
"""
import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import dungeon_maps_b200 as dmap  # noqa: E402
from dungeon_maps_b200 import _params as prm  # noqa: E402
from scripts.time_components import card  # noqa: E402
from scripts.time_egocentric import EPISODE, Walk  # noqa: E402
from scripts.time_reset_envs import make_builder  # noqa: E402
from tests._match import lattice, score_poses as oracle  # noqa: E402

OBSTACLE_HEIGHT = 0.2
WOFF, HOFF = bench.MW / 2., 0.
DYAW = math.radians(1.)


def walk_world(B, C, fixed, dev):
  """World map after steps 0..98 and step 99's local map (camera frame, not merged), with step 99's true pose."""
  walk = Walk(B, C, dev)
  builder = make_builder(dev)
  if fixed:
    builder = dmap.MapBuilder(map_projector=builder.proj, fixed_canvas=(2400, 2400))
  for t in range(EPISODE - 1):
    walk.step(builder, t)
  t = EPISODE - 1
  kw = walk.kw if not C else dict(walk.kw, label_map=walk.labels[t], num_classes=C)
  local = builder.plot(walk.depth[t], cam_pose=walk.poses[t], **kw)
  torch.cuda.synchronize()
  return builder.world_map, local, walk.poses[t].cpu()


def obstacle_free(m):
  seen = m.mask[:, 0]
  obstacle = seen & (m.height_map[:, 0] > OBSTACLE_HEIGHT)
  return obstacle, seen & ~obstacle


def crop_loop(world, planes, window, cands):
  """Arm B: one crop_egocentric_map per candidate."""
  b, C = planes.shape[:2]
  h, w = window.shape[-2:]
  m = dmap.TopdownMap(topdown_map=planes.float(), mask=planes, height_map=None, map_projector=world.proj,
                      is_height_map=True)
  win = window if window.dim() == 4 else window[:, None]
  out = torch.empty((b, C, cands.shape[1]), dtype=torch.int32, device=planes.device)
  for k in range(cands.shape[1]):
    crop = dmap.crop_egocentric_map(m, w, h, cam_pose=cands[:, k], width_offset=WOFF, height_offset=HOFF)
    out[:, :, k] = (crop.mask & win).sum(dim=(2, 3), dtype=torch.int32)
  return out


def per_pass(fn, calls):
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(calls):
      fn()
    torch.cuda.synchronize()
  out = {}
  for ev in prof.key_averages():
    for kernel in ("match_compact_kernel", "match_score_kernel"):
      if kernel in ev.key:
        us = getattr(ev, "device_time_total", None)
        us = ev.cuda_time_total if us is None else us
        out[f"{kernel}_ms"] = round(us / 1e3 / calls, 4)
  return out


def pack_ms(world, cands, hw, dev, calls):
  """Host ms of what score_poses does with the candidates: the blocks packed from torch's sin / cos and uploaded."""
  b, n = cands.shape[:2]
  p = world.proj
  cols = [prm.per_sample(dmap.get(x, 0.), b, ()) for x in (p.width_offset, p.height_offset)]
  cols += [prm.per_sample(WOFF, b, ()), prm.per_sample(HOFF, b, ())]
  ts = []
  for _ in range(calls):
    t0 = time.perf_counter()
    samples = prm.ego_samples(cands.reshape(b * n, 3), *[c[:, None].expand(b, n).reshape(-1) for c in cols], hw)
    blk = prm.upload(samples, dev) if samples.numel() * 4 <= prm._UPLOAD_MAX else \
        samples.pin_memory().to(dev, non_blocking=True)
    ts.append((time.perf_counter() - t0) * 1e3)
    del blk
  torch.cuda.synchronize()
  return float(np.median(ts))


def time_case(name, world, planes, window, true_pose, steps, args, extra):
  dev = planes.device
  b = planes.shape[0]
  planes4 = planes if planes.dim() == 4 else planes[:, None]
  C = planes4.shape[1]
  h, w = window.shape[-2:]
  cands = torch.from_numpy(lattice(true_pose.numpy(), steps, float(world.proj.map_res), DYAW))
  n = cands.shape[1]
  cells = window.reshape(b, -1, h * w).sum(-1).cpu()                    # (b, window planes)
  line = dict(card(), case=name, envs=b, planes=C, world_shape=list(planes.shape[-2:]), window=[h, w],
              window_planes=int(cells.shape[1]), candidates=n, lattice=f"{2 * steps + 1}^3",
              window_true_cells_per_env=cells.sum(1).tolist(),
              window_density=round(float(cells.sum()) / (b * cells.shape[1] * h * w), 4), **extra)

  def call():
    return dmap.score_poses(world, planes, window, cands, width_offset=WOFF, height_offset=HOFF)

  got = call()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.calls):
    call()
  e1.record()
  torch.cuda.synchronize()
  kernel_ms = e0.elapsed_time(e1) / args.calls
  calls = []
  for _ in range(args.calls):
    t0 = time.perf_counter()
    call()
    torch.cuda.synchronize()
    calls.append((time.perf_counter() - t0) * 1e3)
  evals = int(cells.sum()) * n
  line.update(kernel_ms=round(kernel_ms, 4), call_ms_median=round(float(np.median(calls)), 4),
              host_pack_upload_ms_median=round(pack_ms(world, cands, h * w, dev, args.calls), 4),
              cell_candidate_evals=evals, evals_per_s=float(f"{evals / kernel_ms * 1e3:.4g}"),
              plane_tests_per_s=float(f"{evals * (C if cells.shape[1] == 1 else 1) / kernel_ms * 1e3:.4g}"))
  line.update(per_pass(call, args.calls))
  if "match_score_kernel_ms" in line:
    line["score_pass_evals_per_s"] = float(f"{evals / line['match_score_kernel_ms'] * 1e3:.4g}")
  got4 = got if planes.dim() == 4 else got[:, None]
  # arm B
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  want = crop_loop(world, planes4, window, cands)
  torch.cuda.synchronize()
  line["crop_loop_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
  assert torch.equal(got4, want), f"{name}: the crop loop differs"
  # arm C
  subset = np.linspace(0, n - 1, min(args.oracle, n)).round().astype(int)
  t0 = time.perf_counter()
  host = [t.cpu().numpy() for t in (planes4, window if window.dim() == 4 else window[:, None])]
  line["host_copy_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
  p = world.proj
  woff_src = p.width_offset.cpu().numpy() if torch.is_tensor(p.width_offset) else p.width_offset
  hoff_src = p.height_offset.cpu().numpy() if torch.is_tensor(p.height_offset) else p.height_offset
  t0 = time.perf_counter()
  ref = oracle(host[0], host[1], woff_src, hoff_src, p.map_res, p.flip_h, cands[:, subset].numpy(), WOFF, HOFF)
  oracle_ms = (time.perf_counter() - t0) * 1e3
  assert np.array_equal(ref, got4[:, :, subset].cpu().numpy()), f"{name}: the oracle differs"
  line.update(oracle_candidates=len(subset), oracle_ms_per_candidate=round(oracle_ms / len(subset), 1))
  return line, got4


def recipe(world, planes, window, true_pose, line):
  """The docstring's recipe with a known odometry error; reported, not asserted."""
  res = float(world.proj.map_res)
  delta = torch.tensor([3 * res, -2 * res, 3 * DYAW], dtype=torch.float32)
  odom = (true_pose + delta).to(torch.float32)
  cands = torch.from_numpy(lattice(odom.numpy(), 5, res, DYAW))
  s = dmap.score_poses(world, planes, window, cands, width_offset=WOFF, height_offset=HOFF)
  score = (s[:, 0] - s[:, 1]).cpu()
  best = score.argmax(-1)
  b = score.shape[0]
  pose = cands[torch.arange(b), best]
  err = (pose - true_pose).abs()
  within = (err[:, 0] <= res * 1.01) & (err[:, 1] <= res * 1.01) & (err[:, 2] <= DYAW * 1.01)
  nearest = ((cands - true_pose[:, None, :]) / torch.tensor([res, res, DYAW])).abs().amax(-1).argmin(-1)
  top2 = score.float().topk(2, dim=-1).values
  has = window.reshape(b, -1).any(-1).cpu()
  line.update(recipe_odometry_error=[3, -2, 3], recipe_envs_with_obstacle_cells=int(has.sum()),
              recipe_envs_within_one_step=int(within.sum()),
              recipe_envs_within_one_step_among_those=int((within & has).sum()),
              recipe_envs_exact=int((best == nearest).sum()),
              recipe_best_minus_second_min=float((top2[:, 0] - top2[:, 1]).min()),
              recipe_best_minus_second_median=float((top2[:, 0] - top2[:, 1]).median()),
              recipe_best_minus_at_true_max=int((score.max(-1).values - score[torch.arange(b), nearest]).max()),
              recipe_best_minus_at_odometry_median=float((score.max(-1).values - score[:, cands.shape[1] // 2])
                                                         .float().median()),
              recipe_max_error_cells=[round(float(err[:, 0].max()) / res, 2), round(float(err[:, 1].max()) / res, 2)],
              recipe_max_error_deg=round(math.degrees(float(err[:, 2].max())), 2))


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=20)
  ap.add_argument("--oracle", type=int, default=8)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,fixed,semantic")
  args = ap.parse_args()
  if args.calls < 1 or args.oracle < 1:
    ap.error("--calls and --oracle must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_score_poses.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  lines = []

  def emit(line):
    print(json.dumps(line), flush=True)
    lines.append(line)

  for case in args.cases.split(","):
    if case in ("growing", "fixed"):
      world, local, true_pose = walk_world(32, 0, case == "fixed", dev)
      obstacle, free = obstacle_free(world)
      window = obstacle_free(local)[0]
      both = torch.stack((obstacle, free), dim=1)
      jobs = [("obstacle", obstacle, window), ("obstacle+free", both, window),
              ("seen", world.mask[:, 0], local.mask[:, 0])] if case == "growing" else [("fixed", both, window)]
      for name, planes, win in jobs:
        for steps in (5, 2):
          line, _ = time_case(name, world, planes, win, true_pose, steps, args, dict(steps=EPISODE))
          if planes.dim() == 4 and steps == 5:
            recipe(world, planes, window, true_pose, line)
          emit(line)
      del world, local, obstacle, free, window, both
    elif case == "semantic":
      world, local, true_pose = walk_world(8, 16, False, dev)
      planes = world.topdown_map > 0.5
      window = local.topdown_map > 0.5
      for steps in (5, 2):
        emit(time_case("semantic", world, planes, window, true_pose, steps, args, dict(steps=EPISODE))[0])
      del world, local, planes, window
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
