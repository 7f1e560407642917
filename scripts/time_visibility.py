#!/usr/bin/env python
"""visible_cells / count_visible on config-4 world maps: one JSON line per case.

The walk is the one the other time_*.py scripts share (bench.BuilderWorkload geometry over synth room scenes, 480x640
depth -> 400x400 local maps at 3 cm, 100 steps, merged into a global world map).  Obstacle = seen and above 0.2 m;
unknown cells let sight through.  Cases:
  agent window    32 environments, visible_cells from the agent's cell, r = 166 (5 m), on the growing world map and on
                  2400 x 2400 fixed canvases;
  exploration     32 environments, count_visible of the unseen cells from n = 64 lattice candidates around each agent
                  (8 x 8 offsets, 20 cells apart), r = 166, growing world map;
  goal check      8 environments with 16 classes given as class ids, count_visible of the 16 class planes (> 0.5) from
                  the agent's cell, r = 33;
  open map        the growing world's grid with no blockers, so every line is walked in full, visible_cells from the
                  agent's cell at r = 512.
Per case:
  A  the library call: kernel ms from CUDA events around --calls warm calls; call ms, host clock to a device
     synchronise, median; line steps = the sum of m = max(|dx|, |dz|) over the targets in the disk and inside the map
     (from shapes and origins; lines that stop early at a blocker walk fewer), per second of kernel time;
  B  a torch GPU baseline, the same walk as r gathers over every window cell, chunked over origins: ms; equal to A
     bit for bit (asserted);
  C  a device-to-host copy and the numpy oracle (tests/_visibility.py) on --oracle origins: ms per origin (copy
     reported apart); equal to A on those origins (asserted).

usage: python scripts/time_visibility.py [--calls 20] [--oracle 4] [--out results/visibility.jsonl]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dungeon_maps_b200 as dmap  # noqa: E402
from scripts.time_components import card  # noqa: E402
from scripts.time_egocentric import EPISODE, Walk  # noqa: E402
from scripts.time_reset_envs import make_builder  # noqa: E402
from tests import _visibility as oracle  # noqa: E402

OBSTACLE_HEIGHT = 0.2
BASELINE_CHUNK = 1 << 26          # window cells per chunk of the torch baseline


def walk_world(B, C, fixed, dev):
  walk = Walk(B, C, dev)
  builder = make_builder(dev)
  if fixed:
    builder = dmap.MapBuilder(map_projector=builder.proj, fixed_canvas=(2400, 2400))
  for t in range(EPISODE):
    walk.step(builder, t)
  torch.cuda.synchronize()
  return builder.world_map


def torch_visible(blocking, origins, r):
  """Arm B: (b, H, W) bool, (b, n, 2) int64 on the device -> (b, n, 2r+1, 2r+1) bool, the definition as r gathers."""
  b, H, W = blocking.shape
  n = origins.shape[1]
  dev = blocking.device
  side = 2 * r + 1
  d = torch.arange(-r, r + 1, device=dev)
  dz, dx = torch.meshgrid(d, d, indexing="ij")
  ax, az = dx.abs(), dz.abs()
  m, mn = torch.maximum(ax, az), torch.minimum(ax, az)
  sx, sz = torch.where(dx < 0, -1, 1), torch.where(dz < 0, -1, 1)
  xmajor = ax >= az
  disk = dx * dx + dz * dz <= r * r
  flat = blocking.reshape(-1)
  o = origins.reshape(-1, 2)
  out = torch.empty((b * n, side, side), dtype=torch.bool, device=dev)
  step = max(1, BASELINE_CHUNK // (side * side))
  for k0 in range(0, b * n, step):
    k = torch.arange(k0, min(k0 + step, b * n), device=dev)
    ox, oz = o[k, 0][:, None, None], o[k, 1][:, None, None]
    base = (k // n * H * W)[:, None, None]

    def blocked(x, z):
      inside = (x >= 0) & (x < W) & (z >= 0) & (z < H)
      return flat[base + z.clamp(0, H - 1) * W + x.clamp(0, W - 1)] & inside

    tx, tz = ox + dx, oz + dz
    ok = disk & (tx >= 0) & (tx < W) & (tz >= 0) & (tz < H) & (ox >= 0) & (ox < W) & (oz >= 0) & (oz < H)
    px, pz = ox.expand_as(tx), oz.expand_as(tz)
    for i in range(1, r + 1):
      q = (2 * i * mn + m) // (2 * m.clamp(min=1))
      cx = ox + torch.where(xmajor, sx * i, sx * q)
      cz = oz + torch.where(xmajor, sz * q, sz * i)
      diag = (cx != px) & (cz != pz)
      stop = (diag & blocked(cx, pz) & blocked(px, cz)) | ((i < m) & blocked(cx, cz))
      ok &= ~(stop & (i <= m))
      px, pz = cx, cz
    out[k] = ok
  return out.view(b, n, side, side)


def torch_count(visible, targets, origins, r):
  """Arm B, counts: the visible windows against the target planes, (b, C, n) int32."""
  b, n, side, _ = visible.shape
  C, H, W = targets.shape[1:]
  d = torch.arange(-r, r + 1, device=visible.device)
  x = origins[..., 0][:, :, None, None] + d[None, None, None, :]
  z = origins[..., 1][:, :, None, None] + d[None, None, :, None]
  idx = (z.clamp(0, H - 1) * W + x.clamp(0, W - 1)).reshape(b, 1, -1).expand(b, C, -1)
  t = targets.reshape(b, C, H * W).gather(2, idx).view(b, C, n, side, side)
  return (t & visible[:, None]).sum(dim=(3, 4), dtype=torch.int32)


def line_steps(origins, H, W, r):
  """Sum of m = max(|dx|, |dz|) over the targets in the disk and inside the map of every origin inside the map."""
  d = np.arange(-r, r + 1)
  dz, dx = np.meshgrid(d, d, indexing="ij")
  disk = dx * dx + dz * dz <= r * r
  m = np.maximum(np.abs(dx), np.abs(dz))
  total = 0
  for x, z in origins.reshape(-1, 2):
    if 0 <= x < W and 0 <= z < H:
      inside = disk & (x + dx >= 0) & (x + dx < W) & (z + dz >= 0) & (z + dz < H)
      total += int(m[inside].sum())
  return total


def time_case(name, blocking, targets, origins, r, args, extra):
  b, H, W = blocking.shape
  n = origins.shape[1]
  line = dict(card(), case=name, envs=b, origins_per_env=n, radius=r, grid=[H, W],
              planes=0 if targets is None else (targets.shape[1] if targets.dim() == 4 else 1),
              blocking_density=round(float(blocking.float().mean()), 4), **extra)

  def call():
    if targets is None:
      return dmap.visible_cells(blocking, origins, r)
    return dmap.count_visible(blocking, targets, origins, r)

  got = call()
  tg4 = None if targets is None else (targets if targets.dim() == 4 else targets[:, None])
  if tg4 is not None and targets.dim() == 3:
    got = got[:, None]
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
  o_host = origins.cpu().numpy()
  steps = line_steps(o_host, H, W, r)
  line.update(kernel_ms=round(kernel_ms, 4), call_ms_median=round(float(np.median(calls)), 4), line_steps=steps,
              line_steps_per_s=float(f"{steps / kernel_ms * 1e3:.4g}"))
  # arm B
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  vis_b = torch_visible(blocking, origins, r)
  want = vis_b if targets is None else torch_count(vis_b, tg4, origins, r)
  torch.cuda.synchronize()
  line["torch_baseline_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
  del vis_b
  assert torch.equal(got, want), f"{name}: the torch baseline differs"
  # arm C
  t0 = time.perf_counter()
  blk_h = blocking.cpu().numpy()
  tg_h = None if targets is None else tg4.cpu().numpy()
  line["host_copy_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
  picks = [(i % b, (i * 7) % n) for i in range(args.oracle)]
  t0 = time.perf_counter()
  ref = [oracle.visible_window(blk_h[i], int(o_host[i, k, 0]), int(o_host[i, k, 1]), r) for i, k in picks]
  if tg_h is not None:
    ref = [oracle.count_visible(blk_h[i:i + 1], tg_h[i:i + 1], o_host[i:i + 1, k:k + 1], r)[0, :, 0]
           for i, k in picks]
  line.update(oracle_origins=len(picks), oracle_ms_per_origin=round((time.perf_counter() - t0) * 1e3 / len(picks), 1))
  got_h = got.cpu().numpy()
  for (i, k), want_ik in zip(picks, ref):
    have = got_h[i, k] if tg_h is None else got_h[i, :, k]
    assert np.array_equal(have, want_ik), f"{name}: the oracle differs at environment {i}, origin {k}"
  return line


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=20)
  ap.add_argument("--oracle", type=int, default=4)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,fixed,semantic")
  args = ap.parse_args()
  if args.calls < 1 or args.oracle < 1:
    ap.error("--calls and --oracle must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_visibility.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  lines = []

  def emit(line):
    print(json.dumps(line), flush=True)
    lines.append(line)

  for case in args.cases.split(","):
    if case in ("growing", "fixed"):
      world = walk_world(32, 0, case == "fixed", dev)
      seen = world.mask[:, 0]
      obstacle = seen & (world.height_map[:, 0] > OBSTACLE_HEIGHT)
      cam = world.get_camera()[:, None, :]                                   # (b, 1, 2)
      extra = dict(world=case, steps=EPISODE)
      emit(time_case("agent window", obstacle, None, cam, 166, args, extra))
      if case == "growing":
        off = torch.arange(-70, 71, 20, device=dev)
        lattice = torch.stack(torch.meshgrid(off, off, indexing="xy"), dim=-1).reshape(-1, 2)
        emit(time_case("exploration", obstacle, ~seen, cam + lattice[None], 166, args, extra))
        emit(time_case("open map", torch.zeros_like(obstacle), None, cam, 512, args, extra))
      del world, seen, obstacle, cam
    elif case == "semantic":
      world = walk_world(8, 16, False, dev)
      seen = world.mask[:, 0]
      obstacle = seen & (world.height_map[:, 0] > OBSTACLE_HEIGHT)
      planes = world.topdown_map > 0.5
      emit(time_case("goal check", obstacle, planes, world.get_camera()[:, None, :], 33, args,
                     dict(world="growing", steps=EPISODE)))
      del world, seen, obstacle, planes
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
