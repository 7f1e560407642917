#!/usr/bin/env python
"""Semantic MapBuilder steps at BASELINE config-4 geometry (480x640 depth -> 400x400 local maps at 3 cm, the
bench.BuilderWorkload walk) with C one-hot classes: one JSON line per case with ms/step and env-steps/s.

Cases: C step vs general path (native_step=False), float planes (value_map=one_hot) vs class ids
(label_map=, num_classes=), growing world map vs fixed canvas; the two paths of a case run alternately, --repeat times.
Each line also counts the caching allocator's device allocations / frees / retries inside the timed episode.  A second
pass takes per-kernel times of both paths with torch.profiler (CUDA activities).
A semantic world map holds b * C * cells * 9 bytes (values, heights, mask): the default of 8 environments keeps it at a
few GB.

usage: python scripts/time_semantic_builder.py [--envs 8] [--classes 16] [--steps 100] [--warmup STEPS]
                                               [--repeat 2] [--fixed 2400 2400] [--profile-steps 30] [--cases all]
--warmup defaults to one whole episode, as bench.py's builder workloads do: the allocator's cached blocks then serve
the timed episode, as they serve every episode after the first.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
import dungeon_maps_b200 as dmap  # noqa: E402
from dungeon_maps_b200 import synth  # noqa: E402


def card():
  name = torch.cuda.get_device_name(0)
  try:
    limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
  except (OSError, subprocess.SubprocessError):
    limit = "unknown"
  return {"gpu": name, "power_limit": limit or "unknown"}


def make_builder(dev, native, fixed):
  proj = dmap.MapProjector(width=640, height=480, hfov=bench.HFOV, cam_pose=[0., 0., 0.], width_offset=0.,
                           height_offset=0., cam_pitch=bench.PITCH, cam_height=bench.CAM_H, map_res=bench.RES,
                           map_width=bench.MW, map_height=bench.MH, trunc_depth_min=0.15, trunc_depth_max=5.05,
                           clip_border=10, fill_value=dmap.NINF, to_global=True, device=dev)
  return dmap.MapBuilder(map_projector=proj, fixed_canvas=fixed, native_step=native)


class Episode:
  """The walk, its depth frames and a pool of semantic frames (class ids as uint8, and their one-hot planes)."""

  def __init__(self, args, dev):
    self.B, self.C = args.envs, args.classes
    w = bench.BuilderWorkload(argparse.Namespace(scene="room"))
    w.B = self.B
    self.poses = w.walk(self.B, args.steps, 0)
    self.depth = w.frames_for(self.poses, dev, 0)
    pool = min(args.steps, 16)
    self.labels = [synth.block_labels(self.B, self.C, 480, 640, seed=t, device=dev).to(torch.uint8) for t in range(pool)]
    self.onehot = [synth.block_onehot(self.B, self.C, 480, 640, seed=t, device=dev) for t in range(pool)]
    self.local_kw = dict(to_global=False, width_offset=bench.MW / 2., height_offset=0., map_width=bench.MW,
                         map_height=bench.MH)

  def kw(self, t, inputs):
    k = t % len(self.labels)
    sem = dict(value_map=self.onehot[k]) if inputs == "float" else dict(label_map=self.labels[k], num_classes=self.C)
    return dict(self.local_kw, **sem)

  def run(self, builder, inputs, steps):
    builder.reset()
    for t in range(steps):
      builder.step(self.depth[t], cam_pose=self.poses[t], **self.kw(t, inputs))


def time_case(ep, dev, path, inputs, fixed, args):
  builder = make_builder(dev, path == "C", fixed)
  ep.run(builder, inputs, args.warmup)
  builder.reset()
  torch.cuda.synchronize()
  torch.cuda.reset_peak_memory_stats(dev)
  base = torch.cuda.memory_allocated(dev)
  counters = ("num_device_alloc", "num_device_free", "num_alloc_retries")
  before = {k: torch.cuda.memory_stats(dev).get(k, 0) for k in counters}
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  h0 = time.perf_counter()
  e0.record()
  ep.run(builder, inputs, args.steps)
  e1.record()
  torch.cuda.synchronize()
  host_s = time.perf_counter() - h0
  ms = e0.elapsed_time(e1) / args.steps
  after = {k: torch.cuda.memory_stats(dev).get(k, 0) for k in counters}
  wm = builder.world_map
  out = {"case": f"{path} step, {inputs}, {'fixed canvas' if fixed else 'growing world map'}", "path": path,
         "inputs": inputs, "world": "fixed" if fixed else "growing", "envs": ep.B, "classes": ep.C,
         "steps": args.steps, "ms_per_step": round(ms, 4), "env_steps_per_s": round(ep.B / ms * 1e3, 1),
         "host_wall_ms_per_step": round(host_s * 1e3 / args.steps, 4),
         "world_shape_at_end": list(wm.mask.shape),
         "world_bytes_at_end": int(wm.mask.numel()) * 9,
         "peak_allocated_bytes": int(torch.cuda.max_memory_allocated(dev) - base),
         "native_handles": len(builder._handles),
         "warmup_steps": args.warmup,
         **{k: int(after[k] - before[k]) for k in counters}}
  del builder, wm
  return out


def profile_kernels(ep, dev, path, inputs, args):
  """Per-kernel CUDA time of one path over the first profile_steps steps of the walk (growing world map)."""
  from torch.profiler import ProfilerActivity, profile
  builder = make_builder(dev, path == "C", None)
  ep.run(builder, inputs, args.profile_steps)
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    ep.run(builder, inputs, args.profile_steps)
    torch.cuda.synchronize()
  us = defaultdict(float)
  calls = defaultdict(int)
  for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
      us[e.name] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
      calls[e.name] += 1
  fuse = {k: v for k, v in us.items() if "fuse_" in k}
  short = lambda k: k.split("(")[0].replace("void ", "").replace("dm::", "")
  return {"profile": f"{path} step kernels", "path": path, "inputs": inputs, "steps": args.profile_steps,
          "envs": ep.B, "classes": ep.C,
          "merge_us_per_step": round(sum(fuse.values()) / args.profile_steps, 1),
          "all_kernels_us_per_step": round(sum(us.values()) / args.profile_steps, 1),
          "kernels_us_per_step": {short(k): round(v / args.profile_steps, 1)
                                  for k, v in sorted(us.items(), key=lambda kv: -kv[1])},
          "launches_per_step": {short(k): round(calls[k] / args.profile_steps, 2) for k in us}}


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--envs", type=int, default=8)
  ap.add_argument("--classes", type=int, default=16)
  ap.add_argument("--steps", type=int, default=100)
  ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default: --steps)")
  ap.add_argument("--repeat", type=int, default=2)
  ap.add_argument("--fixed", type=int, nargs=2, default=[2400, 2400], metavar=("H", "W"))
  ap.add_argument("--profile-steps", type=int, default=30)
  ap.add_argument("--cases", default="all", help="all | timing | profile")
  args = ap.parse_args()
  if args.warmup is None:
    args.warmup = args.steps
  if args.steps < 1 or args.envs < 1 or not 1 <= args.classes <= 63:
    ap.error("--steps, --envs must be >= 1 and --classes in 1..63")
  if not torch.cuda.is_available():
    sys.exit("time_semantic_builder.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  print(json.dumps(card()), flush=True)
  ep = Episode(args, dev)
  if args.cases in ("all", "timing"):
    for fixed in (None, tuple(args.fixed)):
      for inputs in ("float", "labels"):
        for _ in range(args.repeat):
          for path in ("C", "general"):
            print(json.dumps(time_case(ep, dev, path, inputs, fixed, args)), flush=True)
  if args.cases in ("all", "profile"):
    for inputs in ("float", "labels"):
      for path in ("C", "general"):
        print(json.dumps(profile_kernels(ep, dev, path, inputs, args)), flush=True)


if __name__ == "__main__":
  main()
