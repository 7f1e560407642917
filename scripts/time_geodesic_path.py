#!/usr/bin/env python
"""geodesic_path on config-4 world maps and on a spiral maze: one JSON line per case.

The walk is the one the other time_*.py scripts share (bench.BuilderWorkload geometry over synth room scenes, 480x640
depth -> 400x400 local maps at 3 cm, 100 steps, merged into a global world map).  Traversable = seen and not above
0.2 m, plus the agent's own cell (the agent stands there).  The goal of each environment is its traversable cell
farthest from the agent (the argmax of TopdownMap.geodesic_distance), and dist = geodesic_distance(traversable, goal).
Cases:
  agent path       32 environments, the path from each agent to its goal, max_cells = max(dist) / 5 + 1 (enough for
                   any start), on the growing world map and on 2400 x 2400 fixed canvases;
  waypoints        32 environments, n = 64 starts per environment (the agent's cell plus 8 x 8 lattice offsets 20 cells
                   apart) with max_cells = 256, the waypoint use, growing world map;
  spiral 1024      one 1024 x 1024 one-cell-corridor spiral maze (tests/_geodesic.py), goal in its outer corner, the
                   path from the corridor's inner end, max_cells = its length: the worst case, one serial walk of about
                   half a million cells.
Per case:
  A  the library call: kernel ms from CUDA events around --calls warm calls; call ms, host clock to a device
     synchronise, median; path cells walked (the sum of lengths) per second of kernel time;
  B  a torch GPU loop of one gather step per iteration (the definition over all paths at once, one iteration per path
     cell): ms; equal to A bit for bit (asserted).  Skipped above --torch-max iterations, and the line says so;
  C  a device-to-host copy and the plain-Python oracle walk (tests/_geodesic_path.py) per environment: ms per
     environment (copy reported apart); equal to A (asserted).

usage: python scripts/time_geodesic_path.py [--calls 20] [--torch-max 20000] [--out results/geodesic_path.jsonl]
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
from tests import _geodesic_path as oracle  # noqa: E402
from tests._geodesic import spiral_maze  # noqa: E402

OBSTACLE_HEIGHT = 0.2
# (dx, dz) of the definition's neighbour order, the step costs, and the orthogonal neighbours beside each diagonal one
DIRS = [(dx, dz) for dx, dz, _ in oracle.ORDER]
COSTS = [c for _, _, c in oracle.ORDER]
SIDES = [(k, k) if dx == 0 or dz == 0 else (0 if dx > 0 else 2, 1 if dz > 0 else 3)
         for k, (dx, dz) in enumerate(DIRS)]


def walk_world(B, fixed, dev):
  walk = Walk(B, 0, dev)
  builder = make_builder(dev)
  if fixed:
    builder = dmap.MapBuilder(map_projector=builder.proj, fixed_canvas=(2400, 2400))
  for t in range(EPISODE):
    walk.step(builder, t)
  torch.cuda.synchronize()
  return builder.world_map


def torch_walk(trav, dist, starts, max_cells, max_iters):
  """Arm B: (b, H, W) bool / int32, (b, n, 2) int64 on the device -> (cells, lengths) as geodesic_path, or None past
  max_iters iterations.  Every path takes one step per iteration; liveness is read back every 64 iterations."""
  b, H, W = dist.shape
  n = starts.shape[1]
  dev = dist.device
  D, T = dist.reshape(-1), trav.reshape(-1)
  base = (torch.arange(b * n, device=dev) // n * (H * W))[:, None]
  dx = torch.tensor([d[0] for d in DIRS], device=dev)
  dz = torch.tensor([d[1] for d in DIRS], device=dev)
  cost = torch.tensor(COSTS, device=dev, dtype=torch.int32)
  side_a = torch.tensor([s[0] for s in SIDES], device=dev)
  side_b = torch.tensor([s[1] for s in SIDES], device=dev)
  x, z = starts[..., 0].reshape(-1, 1), starts[..., 1].reshape(-1, 1)

  def read(x, z):
    inside = (x >= 0) & (x < W) & (z >= 0) & (z < H)
    i = base + z.clamp(0, H - 1) * W + x.clamp(0, W - 1)
    return torch.where(inside, D[i], -1), inside & T[i]

  d, t = read(x, z)
  live = d >= 0
  cells = torch.full((b * n, max_cells, 2), -1, dtype=torch.int32, device=dev)
  lengths = torch.zeros((b * n, 1), dtype=torch.int32, device=dev)
  for k in range(max_cells):
    if k >= max_iters:
      return None
    cells[:, k] = torch.where(live, torch.cat([x, z], 1), -1).to(torch.int32)
    lengths += live.to(torch.int32)
    go = live & (d > 0) & t & (k + 1 < max_cells)
    qx, qz = x + dx, z + dz                                        # (P, 8)
    dq, tq = read(qx, qz)
    ok = go & (dq >= 0) & (dq == d - cost) & (tq[:, side_a] & tq[:, side_b] | (side_a == side_b))
    moved = ok.any(1, keepdim=True)
    first = ok.to(torch.int8).argmax(1, keepdim=True)               # the first qualifying neighbour in the order
    x = torch.where(moved, qx.gather(1, first), x)
    z = torch.where(moved, qz.gather(1, first), z)
    d = torch.where(moved, dq.gather(1, first), d)
    t = torch.where(moved, tq.gather(1, first), t)
    live = moved
    if k % 64 == 63 and not bool(live.any()):
      break
  return cells.view(b, n, max_cells, 2), lengths.view(b, n)


def time_case(name, trav, dist, starts, max_cells, args, extra):
  b, H, W = dist.shape
  n = starts.shape[1]
  line = dict(card(), case=name, envs=b, starts_per_env=n, grid=[H, W], max_cells=max_cells, **extra)

  def call():
    return dmap.geodesic_path(trav, dist, starts, max_cells)

  cells, lengths = call()
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
  walked = int(lengths.sum())
  line.update(cells_walked=walked, path_len_max=int(lengths.max()),
              path_len_mean=round(float(lengths.float().mean()), 1), output_mb=round(cells.numel() * 4 / 2 ** 20, 1), kernel_ms=round(kernel_ms, 4),
              call_ms_median=round(float(np.median(calls)), 4),
              cells_per_s=float(f"{walked / kernel_ms * 1e3:.4g}"))
  # arm B
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  got = torch_walk(trav, dist, starts, max_cells, args.torch_max)
  torch.cuda.synchronize()
  if got is None:
    line.update(torch_loop_ms=None, torch_loop="not run: more than --torch-max iterations")
  else:
    line["torch_loop_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    assert torch.equal(got[0], cells) and torch.equal(got[1], lengths), f"{name}: the torch loop differs"
  del got
  # arm C
  t0 = time.perf_counter()
  th, dh = trav.cpu().numpy(), dist.cpu().numpy()
  line["host_copy_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
  sh = starts.cpu().numpy()
  t0 = time.perf_counter()
  want = [oracle.oracle(th[i:i + 1], dh[i:i + 1], sh[i:i + 1], max_cells) for i in range(b)]
  line["oracle_ms_per_env"] = round((time.perf_counter() - t0) * 1e3 / b, 1)
  got_c, got_l = cells.cpu().numpy(), lengths.cpu().numpy()
  for i, (wc, wl) in enumerate(want):
    assert np.array_equal(got_l[i], wl[0]) and np.array_equal(got_c[i], wc[0]), f"{name}: the oracle differs at {i}"
  return line


def world_case(fixed, dev):
  """(traversable, dist, agent cells (b, 1, 2)) of a 32-environment config-4 walk."""
  world = walk_world(32, fixed, dev)
  free = world.mask[:, 0] & (world.height_map[:, 0] <= OBSTACLE_HEIGHT)
  b, H, W = free.shape
  cam = world.get_camera()
  free[torch.arange(b, device=dev), cam[:, 1], cam[:, 0]] = True
  far = world.geodesic_distance(free).flatten(1).argmax(1)
  dist = dmap.geodesic_distance(free, torch.stack([far % W, far // W], -1))
  del world
  return free, dist, cam[:, None, :]


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=20)
  ap.add_argument("--torch-max", type=int, default=20000)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,fixed,spiral")
  args = ap.parse_args()
  if args.calls < 1:
    ap.error("--calls must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_geodesic_path.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  lines = []

  def emit(line):
    print(json.dumps(line), flush=True)
    lines.append(line)

  for case in args.cases.split(","):
    if case in ("growing", "fixed"):
      free, dist, cam = world_case(case == "fixed", dev)
      extra = dict(world=case, steps=EPISODE, traversable_share=round(float(free.float().mean()), 4))
      emit(time_case("agent path", free, dist, cam, int(dist.max()) // 5 + 1, args, extra))
      if case == "growing":
        off = torch.arange(-70, 71, 20, device=dev)
        lattice = torch.stack(torch.meshgrid(off, off, indexing="xy"), dim=-1).reshape(-1, 2)
        starts = torch.cat([cam, cam + lattice[None, 1:]], dim=1)         # the agent first, 64 starts in all
        emit(time_case("waypoints", free, dist, starts, 256, args, extra))
      del free, dist, cam
    elif case == "spiral":
      N = 1024
      trav = torch.from_numpy(spiral_maze(N, N)[None]).to(dev)
      dist = dmap.geodesic_distance(trav, torch.tensor([[[0, 0]]]))
      far = int(dist.flatten().argmax())
      start = torch.tensor([[[far % N, far // N]]], device=dev)
      emit(time_case("spiral 1024", trav, dist, start, int(dist.max()) // 5 + 1, args,
                     dict(traversable_share=round(float(trav.float().mean()), 4))))
      del trav, dist
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
