#!/usr/bin/env python
"""Benchmark of the render path: forward + backward of render_gaussians on synthetic gaussians.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json metric "fwd+bwd ms/frame & Gaussians*px/s at 3M Gauss 2048px"): 3,000,000 seeded random
gaussians (taichi_splatting/tests/random_data.py recipe), spherical harmonics degree 3, 2048x1365, tile 16.
A step is one batch of `views_per_rank` camera views per rank, forward + backward through the public API
(render_gaussians -> L1 loss -> backward), gradients accumulated over the views, then ONE gradient all-reduce
(NCCL) when N > 1.  Gaussians are replicated on every rank, views are partitioned (weak scaling: per-GPU work
is fixed).  value = gaussians * pixels * views of all ranks / second.

Prints ONE JSON line (see the keys below).  `--impl reference` times the CPU restatement of the reference
algorithm (oracle/) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# The CPU legs (cpu_baseline, --impl reference) render the SAME scene at FULL size: same 3 M gaussians, camera and
# resolution as the GPU arm (BASELINE.md §3: full size whenever a frame takes under a minute; it takes a few seconds).
WORKLOADS = {
  # BASELINE.json metric: "fwd+bwd ms/frame & Gaussians*px/s at 3M Gauss 2048px"
  "bench": dict(scene="bench", tile_size=16, seed=0),
  # BASELINE.json config 5: batched multi-view step, 64 cameras x 3 M gaussians at 1600x1064 (use --total-views 64)
  "c5": dict(scene="c5", tile_size=16, seed=0),
}


# ----------------------------------------------------------------------------------------------- scene
def build_scene(scene, seed, num_views, num_gaussians=None, image_size=None):
  """The scene of a BASELINE.json configuration (synthetic.baseline_scene) and `num_views` cameras: the scene's own
  camera first, then small pose jitters around it so that every view sees a comparable part of the scene."""
  from taichi_gaussian_rasterizer_b200.synthetic import baseline_scene
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import join_rt, quat_to_mat
  gaussians, base, spec = baseline_scene(scene, seed=seed, n=num_gaussians or None, image_size=image_size)
  cameras = []
  g = torch.Generator().manual_seed(seed + 1)
  for i in range(num_views):
    axis = torch.nn.functional.normalize(torch.randn(3, generator=g), dim=0)
    angle = (torch.rand(1, generator=g) * 2 - 1) * 0.02
    q = torch.cat([axis * torch.sin(angle / 2), torch.cos(angle / 2)])
    delta = join_rt(quat_to_mat(q), (torch.rand(3, generator=g) * 2 - 1) * 0.02)
    cameras.append(base.transformed(delta) if i > 0 else base)
  return gaussians, cameras, spec


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
  """SM clock + throttle reasons sampled DURING the timed region (NVML in a thread, every 20 ms; nvidia-smi as a
  fallback when pynvml is unavailable)."""
  REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

  def __init__(self, index):
    self.index, self.sm, self.mask, self.max_mhz = index, [], 0, None
    self._stop = threading.Event()
    self.thread = None
    self.source = None

  def _loop_nvml(self, nvml, handle):
    while not self._stop.is_set():
      try:
        self.sm.append(float(nvml.nvmlDeviceGetClockInfo(handle, nvml.NVML_CLOCK_SM)))
        self.mask |= int(nvml.nvmlDeviceGetCurrentClocksEventReasons(handle))
      except Exception:
        pass
      self._stop.wait(0.02)

  def _loop_smi(self):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
    while not self._stop.is_set():
      try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             stdout=subprocess.PIPE, text=True, timeout=5).stdout.strip().split(",")
        self.sm.append(float(out[0])); self.max_mhz = float(out[1]); self.mask |= int(out[2].strip(), 16)
      except Exception:
        pass
      self._stop.wait(0.05)

  def start(self):
    try:
      import pynvml as nvml
      nvml.nvmlInit()
      visible = os.environ.get("CUDA_VISIBLE_DEVICES")
      phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
      handle = nvml.nvmlDeviceGetHandleByIndex(phys)
      self.max_mhz = float(nvml.nvmlDeviceGetMaxClockInfo(handle, nvml.NVML_CLOCK_SM))
      self.thread = threading.Thread(target=self._loop_nvml, args=(nvml, handle), daemon=True)
      self.source = "nvml"
    except Exception:
      self.thread = threading.Thread(target=self._loop_smi, daemon=True)
      self.source = "nvidia-smi"
    self.thread.start()

  def stop(self):
    if self.thread is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampler not started"], "samples": 0}
    self._stop.set()
    self.thread.join(timeout=6)
    sm = sorted(self.sm)
    reasons = sorted(n for n, bit in self.REASONS.items() if self.mask & bit)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
            "samples": len(sm), "source": self.source}


# ----------------------------------------------------------------------------------------------- ours
KERNELS_PER_CALL = {  # kernels launched by each entry point (memsets not counted)
  "gs_project_fwd": 1, "gs_project_bwd": 1, "gs_sh_fwd": 1, "gs_sh_bwd": 1, "gs_tile_count": 1, "gs_full_cumsum": 1,
  "gs_tile_emit_keys": 1, "gs_find_ranges": 1, "gs_raster_fwd": 2, "gs_raster_bwd": 2,
  "gs_depth_keys": 1, "gs_tile_count_perm": 1, "gs_tile_emit_tiles": 1, "gs_find_ranges_tiles": 1,
  "gs_camera_position": 1, "gs_sh_fwd_counted": 1, "gs_sh_bwd_stage": 1, "gs_sh_bwd_flush": 1,
  "gs_sh_fwd_views": 1, "gs_gather_rows_counted": 1, "gs_depth_keys_counted": 1, "gs_tile_count_perm_counted": 1,
  "gs_full_cumsum_counted": 1,
}


def resolve_workload(args):
  """(workload dict, views per rank, scaling) from the command line: `--workload bench` (default; weak scaling, a fixed
  number of views per rank) or `--workload c5 --total-views 64` (BASELINE config 5: the batch is fixed and split over
  the ranks = strong scaling)."""
  from taichi_gaussian_rasterizer_b200.synthetic import BASELINE_SCENES
  W = dict(WORKLOADS[args.workload])
  spec = dict(BASELINE_SCENES[W["scene"]])
  W.update(num_gaussians=args.num_gaussians or spec["n"], image_size=tuple(args.image_size or spec["image_size"]),
           sh_degree=spec["sh_degree"], scale_factor=spec.get("scale_factor", 1.0))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  if args.total_views:
    assert args.total_views % world == 0, f"--total-views {args.total_views} does not divide over {world} ranks"
    return W, args.total_views // world, "strong"
  return W, args.views_per_rank, "weak"


def workload_name(W):
  w, h = W["image_size"]
  return (f"render_gaussians fwd+bwd, {W['num_gaussians']} random gaussians, SH degree {W['sh_degree']}, "
          f"{w}x{h}, tile {W['tile_size']}, L1 loss")


def run_ours(args):
  import torch.distributed as dist
  from taichi_gaussian_rasterizer_b200 import RasterConfig, _native, evaluate_sh_views, render_gaussians
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket, run_views
  from taichi_gaussian_rasterizer_b200.perspective import CameraParams

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
  torch.cuda.set_device(local_rank)
  device = torch.device("cuda", local_rank)
  if world > 1:
    dist.init_process_group("nccl", device_id=device)

  W, views, scaling = resolve_workload(args)
  w, h = W["image_size"]
  gaussians_cpu, cameras, _ = build_scene(W["scene"], W["seed"], views * world, W["num_gaussians"], W["image_size"])
  my_cameras = cameras[rank::world][:views]
  gaussians = gaussians_cpu.to(device=device)
  if args.morton:
    # one-off scene preparation, outside the timed region: rows of every tensor permuted into Morton order of the
    # positions (misc/morton_sort.py) — same gaussians, same images, neighbours in space adjacent in memory
    from taichi_gaussian_rasterizer_b200.misc import morton_sort
    extent = (gaussians.position.max(dim=0).values - gaussians.position.min(dim=0).values).max().item()
    order = morton_sort.argsort(gaussians.position.contiguous(), extent / 2 ** 20).long()
    gaussians = gaussians.apply(lambda t: t[order].contiguous(), batch_size=gaussians.batch_size)
  gaussians.requires_grad_(True)
  params = [gaussians.position, gaussians.log_scaling, gaussians.rotation, gaussians.alpha_logit, gaussians.feature]
  # N > 1: the bucket lives in symmetric memory with an NVSwitch multicast mapping and is summed by our own kernel
  # (csrc/multimem_reduce.cu) on the step's streams, inside the step's CUDA graph; --nccl-bucket = ncclAllReduce
  # Measured (gpurun_out/s8_*): 8 GPUs 21.22 ms per step against 21.37 with NCCL; 2 GPUs 21.30 against 20.59 — through
  # the switch (1 + 1/N) x the bucket crosses each link, a two-GPU exchange moves 1 x: used from four ranks up.
  bucket = GradientBucket(params, symmetric=(world >= args.symmetric_from and args.symmetric))
  bucket.pipeline_chunks = args.pipeline_chunks
  if world > 1 and args.reduce_early and args.background_ctas > 0:
    from taichi_gaussian_rasterizer_b200.distributed import make_background_group
    bucket.background_group = make_background_group(args.background_ctas)
  config = RasterConfig(tile_size=W["tile_size"])

  # per step inputs: camera (projection + pose) and the target image of every view, in pinned host memory
  torch.manual_seed(1234 + rank)
  # target images live on the host as a trainer holds them: 8 bit RGB (a dataset image), converted to float on the device
  host_targets = [torch.randint(0, 256, (h, w, 3), dtype=torch.uint8).pin_memory() for _ in range(views)]
  # f32, contiguous, pinned: a copy that converts or gathers on the way goes through an unpinned temporary (and cannot
  # be captured in a CUDA graph)
  host_proj = [c.projection.detach().to(torch.float32).contiguous().clone().pin_memory() for c in my_cameras]
  host_pose = [c.T_camera_world.detach().to(torch.float32).contiguous().clone().pin_memory() for c in my_cameras]
  dev_targets = [t.to(device).to(torch.float32).mul_(1.0 / 255.0) for t in host_targets]
  dev_cams = [c.to(device=device) for c in my_cameras]
  h2d_bytes = sum(t.numel() for t in host_targets) + sum(p.numel() * 4 for p in host_proj + host_pose)
  # the step's result (its loss) is read on the host one step late, from the slot the previous step filled: the host
  # never drains the stream inside the timed region, every step still delivers its 4 bytes
  loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
  loss_ready = [torch.cuda.Event() for _ in range(2)]
  losses_read = []
  stats = {"e2e_step": 0}

  graph_state = {"capacity": None, "totals": None, "graphs": {}, "error": None, "capturing": False}

  def step(from_host: bool, static: bool = False, collective: bool = True):
    with bucket.fused_accumulation():
      return _step(from_host, static, collective)

  copy_stream = torch.cuda.Stream(device=device)
  staged = [dict(target=torch.empty(h, w, 3, dtype=torch.uint8, device=device), proj=torch.empty(4, device=device),
                 pose=torch.empty(4, 4, device=device), ready=torch.cuda.Event(), free=torch.cuda.Event())
            for _ in range(views)]

  poses_ready = torch.cuda.Event()
  # high-priority view streams: the library launches the two big rasterizer kernels at the LOWEST priority whatever the
  # stream's (csrc/common.cuh launch_background), so every other kernel of a view gets SM room first and runs under the
  # other views' rasterizers
  view_streams = ([torch.cuda.Stream(device=device, priority=args.stream_priority) for _ in range(args.streams)]
                  if args.streams > 1 else [])
  if args.kernel_variant:
    from taichi_gaussian_rasterizer_b200 import set_raster_options
    set_raster_options(kernel_variant=args.kernel_variant)

  phase_events = []   # per timed device step: events around [reduce_early | last view | all_reduce]

  def _step(from_host: bool, static: bool = False, collective: bool = True):
    """static: every view through render_gaussians(..., overlap_capacity=) — nothing is read back, the step can be
    captured in a CUDA graph; collective=False: stop after the flush of the deferred SH gradient (the all-reduce is
    issued by the caller, outside the graph)."""
    phase = phase_events if (stats.get("record_phases") and world > 1 and not static) else None   # the markers join the view streams
    compute = torch.cuda.current_stream(device)
    capturing = graph_state["capturing"]
    if from_host:
      # this step's inputs (camera + target image of every view) go host -> device on a side stream: the (tiny) camera
      # blocks of all views first, then the target images, so the copy of view i+1's image overlaps the rendering of
      # view i; the compute stream waits on each event before using what it guards
      if capturing:
        copy_stream.wait_stream(compute)          # the copy stream joins the capture; replays are ordered on `compute`
      with torch.cuda.stream(copy_stream):
        for i in range(views):
          st = staged[i]
          if not capturing:
            copy_stream.wait_event(st["free"])    # the previous step has finished reading this slot
          st["proj"].copy_(host_proj[i], non_blocking=True)
          st["pose"].copy_(host_pose[i], non_blocking=True)
        poses_ready.record(copy_stream)
        for i in range(views):
          st = staged[i]
          st["target"].copy_(host_targets[i], non_blocking=True)
          st["ready"].record(copy_stream)
      compute.wait_event(poses_ready)
      cams = [CameraParams(projection=st["proj"], T_camera_world=st["pose"], near_plane=my_cameras[i].near_plane,
                           far_plane=my_cameras[i].far_plane, image_size=my_cameras[i].image_size)
              for i, st in enumerate(staged)]
    else:
      cams = dev_cams
    bucket.zero_()
    # the batch's cameras are known up front: the SH coefficients are read once for all views of the step
    colors = (evaluate_sh_views(gaussians.feature, gaussians.position, [c.camera_position for c in cams])
              if args.batched_sh else [None] * views)
    # Views are independent until their gradients meet in the bucket: distributed.run_views issues them round robin
    # on `--streams` CUDA streams (the backward of one view runs under the read-backs of the next view's forward)
    def before_last():
      if phase is not None:
        phase.append([torch.cuda.Event(enable_timing=True) for _ in range(4)])
        phase[-1][0].record()
      if views > 1 and args.reduce_early:
        bucket.reduce_early()   # N > 1: the SH slices are all-reduced under the last view (distributed.py)
      if phase is not None:
        phase[-1][1].record()

    def one_view(i):
      extra = dict(overlap_capacity=graph_state["capacity"], overlap_total_out=graph_state["totals"][i]) if static else {}
      rendering = render_gaussians(gaussians, cams[i], config, use_sh=True, sh_colors=colors[i], **extra)
      if from_host:   # the target image is only needed by the loss: its copy runs under the view's forward pass
        st = staged[i]
        torch.cuda.current_stream(device).wait_event(st["ready"])
        target = st["target"].to(torch.float32).mul_(1.0 / 255.0)   # two small elementwise kernels, inside the timed region
      else:
        target = dev_targets[i]
      loss = torch.nn.functional.l1_loss(rendering.image, target)   # mean |image - target|, one fused ATen op each way
      loss.backward()
      if from_host and not capturing:
        st["free"].record(torch.cuda.current_stream(device))
      stats["V"] = rendering.points_in_view.shape[0]
      return loss.detach()

    need_hook = (phase is not None or (world > 1 and views > 1 and args.reduce_early)) and \
      (not static or bucket.reducer is not None)
    total = run_views(views, one_view, view_streams, before_last if need_hook else None)
    if phase is not None:
      phase[-1][2].record()
    if collective:
      bucket.all_reduce()
    else:
      bucket.flush()
    if phase is not None:
      phase[-1][3].record()
    if from_host and not capturing:
      k = stats["e2e_step"]
      slot = k & 1
      loss_host[slot].copy_(total.reshape(1), non_blocking=True)
      loss_ready[slot].record(compute)
      if k > 0:   # read the PREVIOUS step's loss: it has long arrived, the host does not wait for this step's work
        loss_ready[slot ^ 1].synchronize()
        losses_read.append(float(loss_host[slot ^ 1].item()))
      stats["e2e_step"] = k + 1
    return total

  def stock_step():
    """The reference's call sequence, nothing else: render_gaussians(use_sh=True) per view (per view SH evaluation),
    plain autograd accumulation into .grad (no bucket sinks, no deferred SH gradient, no batched colours)."""
    for p in params:
      p.grad = None
    for i in range(views):
      rendering = render_gaussians(gaussians, dev_cams[i], config, use_sh=True)
      torch.nn.functional.l1_loss(rendering.image, dev_targets[i]).backward()

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def timed(fn, steps, timer=None):
    barrier()
    _native.set_stage_timer(timer)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
      fn()
    b.record()
    barrier()
    _native.set_stage_timer(None)
    ms = a.elapsed_time(b)
    if world > 1:
      t = torch.tensor([ms], device=device)
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    return ms

  # ---- the step as ONE CUDA graph (default): every view runs through render_gaussians(..., overlap_capacity=), which
  # reads nothing back, so the ~370 launches of a step (two view streams as parallel branches, H2D copies included in
  # the end-to-end variant) are replayed by one cudaGraphLaunch; the gradient all-reduce (N > 1) follows the replay.
  def capture(from_host: bool):
    from taichi_gaussian_rasterizer_b200 import CapturedStep
    graph_state["capturing"] = True    # _step: no waits on events of earlier eager steps (also during the warm-up runs)
    try:
      captured = CapturedStep(lambda: step(from_host, static=True, collective=in_graph_collective), device=device)
    finally:
      graph_state["capturing"] = False
    return captured.graph, {"total": captured.result, "captured": captured}

  def graph_step(from_host: bool):
    g, holder = graph_state["graphs"][from_host]
    g.replay()
    if world > 1 and not in_graph_collective:
      bucket.all_reduce()   # nothing pending: one all-reduce of the flat bucket
    if from_host:
      k = stats["e2e_step"]
      slot = k & 1
      loss_host[slot].copy_(holder["total"].reshape(1), non_blocking=True)
      loss_ready[slot].record(torch.cuda.current_stream(device))
      if k > 0:
        loss_ready[slot ^ 1].synchronize()
        losses_read.append(float(loss_host[slot ^ 1].item()))
      stats["e2e_step"] = k + 1
    return holder["total"]

  # our multimem reduction is a kernel on the step's streams: it is captured with the step; NCCL's follows the replay
  in_graph_collective = bucket.reducer is not None
  use_graph, graph_check = False, None
  if args.graph:
    try:
      from taichi_gaussian_rasterizer_b200 import overlap_capacity_for
      graph_state["capacity"] = overlap_capacity_for(gaussians, dev_cams, config)
      graph_state["totals"] = [torch.zeros(1, dtype=torch.int32, device=device) for _ in range(views)]
      step(False)
      eager_flat = bucket.flat.clone()
      graph_state["graphs"][False] = capture(False)
      graph_state["graphs"][True] = capture(True)
      graph_step(False)
      torch.cuda.synchronize()
      # the replayed step against the eager default path (same kernels; sums differ by the order of the atomic adds)
      graph_check = float(((bucket.flat.double() - eager_flat.double()).norm() / eager_flat.double().norm()).item())
      del eager_flat
      use_graph = True
    except Exception as e:   # noqa: BLE001 - report and fall back to the eager step
      import traceback
      traceback.print_exc(file=sys.stderr)
      graph_state["error"] = f"{type(e).__name__}: {e}"[:300]
      graph_state["graphs"].clear()
      graph_state["capturing"] = False
      torch.cuda.synchronize()
  last = {}

  def run_dev():
    last["loss"] = graph_step(False) if use_graph else step(False)

  run_e2e = (lambda: graph_step(True)) if use_graph else (lambda: step(True))

  for _ in range(args.warmup):
    run_dev()
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  stats["record_phases"] = True
  ms_dev = timed(run_dev, args.steps)
  stats["record_phases"] = False
  # the passes below run the step again and overwrite the bucket: the last timed step's outputs are copied out now
  dumped = None
  if args.dump_outputs and rank == 0:
    names = ("position", "log_scaling", "rotation", "alpha_logit", "feature")
    dumped = sample_outputs(last["loss"], {k: p.grad for k, p in zip(names, params)})
  ms_eager = None
  if use_graph and world == 1:   # the same step issued eagerly (round 2a's headline), for the record
    for _ in range(2):
      step(False)
    ms_eager = timed(lambda: step(False), max(2, args.steps // 2)) / max(2, args.steps // 2)
  ms_no_stale = None
  if use_graph and world == 1 and not args.no_stock:
    # for the record: the same graph step WITHOUT the reference's stale-slot re-read (SURVEY Q1: tiles with more than
    # 256 overlaps blend up to 255 gaussians of the previous group a second time; emulate_stale_tail reproduces it and
    # is what every parity claim and the headline are measured with)
    from taichi_gaussian_rasterizer_b200 import set_raster_options
    saved_graph = graph_state["graphs"][False]
    try:
      set_raster_options(emulate_stale_tail=False)
      graph_state["graphs"][False] = capture(False)
      for _ in range(2):
        graph_step(False)
      ms_no_stale = timed(lambda: graph_step(False), max(2, args.steps // 2)) / max(2, args.steps // 2)
    except Exception:   # noqa: BLE001 - an extra, never fatal
      ms_no_stale = None
    finally:
      set_raster_options(emulate_stale_tail=True)
      graph_state["graphs"][False] = saved_graph
  # per entry point device times (CUDA events on the launching stream) come from a SECOND pass with the views issued one
  # after another on one stream: with two view streams a kernel shares the SMs with the other view's kernels and its
  # event-to-event time is not the kernel's own (the roofline wants the kernel timed alone)
  timer = _native.StageTimer()
  saved_streams = list(view_streams)
  view_streams.clear()
  stage_steps = max(2, args.steps // 2)
  for _ in range(2):   # the current stream's allocator pool has to grow first (the view streams own the cached blocks)
    step(False)
  ms_single = timed(lambda: step(False), stage_steps, timer)
  view_streams.extend(saved_streams)
  stage = timer.summary()
  # where the end of a step goes on this rank (device time, averaged over the timed steps): flushing + launching the
  # early reduction, the last view (which shares the SMs with that reduction when N > 1), the closing all_reduce()
  phase_ms = {name: sum(e[i].elapsed_time(e[i + 1]) for e in phase_events) / max(len(phase_events), 1)
              for i, name in enumerate(("reduce_early_launch", "last_view", "all_reduce_tail"))}
  clocks = sampler.stop() if rank == 0 else None
  run_e2e()
  ms_e2e = timed(run_e2e, args.steps)
  overlap_total_max = None
  if use_graph:
    overlap_total_max = max(int(t.item()) for t in graph_state["totals"])
    assert overlap_total_max <= graph_state["capacity"], "overlap capacity exceeded: the timed images dropped gaussians"
  stock_ms = None
  if world == 1 and not args.no_stock:
    saved = [p.grad for p in params]
    stock_steps = max(2, min(args.steps, 5))
    stock_step()
    stock_ms = timed(stock_step, stock_steps) / stock_steps / views
    for p, gr in zip(params, saved):   # the bucket's views back in place
      p.grad = gr

  n, px = W["num_gaussians"], w * h
  units_per_step = n * px * views * world
  value = units_per_step / (ms_dev / args.steps / 1e3)
  e2e = units_per_step / (ms_e2e / args.steps / 1e3)

  # K of the first view, for the roofline's algorithmic bytes
  from taichi_gaussian_rasterizer_b200 import map_to_tiles
  from taichi_gaussian_rasterizer_b200.perspective.projection import project_to_image
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import ndc_depth
  with torch.no_grad():
    g2d, depths, idx = project_to_image(gaussians, dev_cams[0], config)
    o2p, ranges = map_to_tiles(g2d, ndc_depth(depths, dev_cams[0].near_plane, dev_cams[0].far_plane),
                               dev_cams[0].image_size, config)
  V, K, F = int(idx.shape[0]), int(o2p.shape[0]), 3
  counts = (ranges[..., 1] - ranges[..., 0]).float()

  peaks = {}
  try:
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
  except Exception:
    pass
  peak_gbs, peak_src = (peaks["hbm_gbs"], "MEASURED_PEAKS.json") if "hbm_gbs" in peaks else (6650.0, "fallback")
  traffic, traffic_src, warp_inst = None, None, None
  try:   # dram bytes per launch of the dominant kernel, from the committed `ncu --set full` capture of this workload
    t = json.loads((ROOT / "profiles" / "roofline_traffic.json").read_text())["raster_bwd_fast_kernel"]
    traffic, traffic_src = t["dram_bytes_per_launch"], t["source"]
    warp_inst = t.get("warp_instructions_per_launch")
  except Exception:
    pass
  calls, bwd_ms = stage.get("gs_raster_bwd", (0, 0.0))
  bwd_avg_ms = bwd_ms / max(calls, 1)
  bwd_bytes = K * (32 + 4 * F) + 8 * px * F + V * (28 + 4 * F)   # SURVEY.md §8(d) raster_bwd
  achieved = bwd_bytes / (bwd_avg_ms * 1e-3) / 1e9 if bwd_avg_ms > 0 else 0.0
  # the kernel is issue bound: warp instructions per launch (ncu smsp__inst_executed.sum, same capture) over the live
  # launch time, against 148 SMs x 4 schedulers x the SM clock sampled during the run
  issue = None
  if warp_inst and bwd_avg_ms > 0:
    sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    peak_ips = 148 * 4 * sm_mhz * 1e6
    ach_ips = warp_inst / (bwd_avg_ms * 1e-3)
    issue = {"warp_inst_per_launch": warp_inst, "achieved_warp_inst_per_s": ach_ips, "peak_warp_inst_per_s": peak_ips,
             "frac": ach_ips / peak_ips, "source": traffic_src}
  stage_ms = {k: round(v[1] / stage_steps / views, 4) for k, v in sorted(stage.items())}
  launches = sum(KERNELS_PER_CALL.get(k, 0) * v[0] for k, v in stage.items())
  # two sorts per frame, each = histogram + one kernel per digit pass: the depth keys (32 bits, enqueued with
  # the count still on the device: gs_radix_sort_pairs_counted) and the tile ids (tile_bits)
  tile_bits = max(1, (int(ranges.shape[0] * ranges.shape[1]) - 1).bit_length())
  launches += stage.get("gs_radix_sort_pairs_counted", (0, 0.0))[0] * (1 + 4)
  launches += stage.get("gs_radix_sort_pairs", (0, 0.0))[0] * (1 + -(-tile_bits // 8))
  launches = launches // max(stage_steps, 1)

  # HBM rooflines of the bandwidth-bound stages: SURVEY.md §8(d) algorithmic bytes per launch over the live CUDA-event
  # time of the entry point (the sort figure covers both sorts of a frame: V depth keys in 4 passes, K tile ids in 2)
  T_tiles, CD = int(ranges.shape[0] * ranges.shape[1]), 3 * (W["sh_degree"] + 1) ** 2
  passes_k = -(-tile_bits // 8)
  alg_bytes = {
    "gs_project_fwd": 44 * n + 40 * V,
    "gs_project_bwd": 84 * V + 44 * n + 44 * V,                 # + the read half of the in-kernel accumulation
    "gs_sh_fwd_counted": V * (8 + 12 + 4 * CD) + 12 * V,
    "gs_sh_bwd": V * (32 + 12) + 4 * CD * n + 4 * CD * V,        # coefficient rows not read; bucket rows read + written
    # deferred SH gradient: per view the masked colour gradient is staged (V x (out, grad, index) in, (N,3) out) ...
    "gs_sh_bwd_stage": V * (12 + 12 + 8) + 12 * n,
    # batched SH colours: coefficient rows + positions read once per step, (N,3) written per view (per frame share);
    # a view gathers its visible rows
    "gs_sh_fwd_views": (n * (4 * CD + 12 + 12 * views)) // views,
    "gs_gather_rows_counted": V * (8 + 12 + 12),
    # ... and one flush per step reads the staged views + positions and adds to the coefficient rows (per frame share)
    "gs_sh_bwd_flush": (n * (12 * views + 12 + 4 * CD)) // views,   # rows written, not read: zero_() marked them clean
    "gs_full_cumsum": 8 * V,
    "gs_full_cumsum_counted": 8 * V,
    "gs_tile_emit_tiles": 20 * V + 8 * K,
    "gs_radix_sort_pairs_counted": 4 * V + 16 * V * 4,          # depth keys: histogram read + 4 passes over 8 B pairs
    "gs_radix_sort_pairs": 4 * K + 16 * K * passes_k,            # tile ids
    "gs_find_ranges_tiles": 4 * K + 8 * T_tiles,
  }
  hbm_stages = {}
  for name, nbytes in alg_bytes.items():
    ms = stage_ms.get(name)
    if ms:
      gbs = nbytes / (ms * 1e-3) / 1e9
      hbm_stages[name] = {"algorithmic_bytes": int(nbytes), "ms": ms, "achieved_gbs": round(gbs, 1),
                          "frac": round(gbs / peak_gbs, 3) if peak_gbs else None}

  out = {
    "metric": "gaussians_px_per_s_fwd_bwd", "value": value, "unit": "gaussian*pixel/s",
    "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
    "ms_per_step": ms_dev / args.steps, "ms_per_frame": ms_dev / args.steps / views,
    "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    "config": {"workload": workload_name(W),
               "views_per_rank": views, "view_streams": max(args.streams, 1), "view_stream_priority": args.stream_priority, "parallelism": f"view-parallel x{world}, replicated gaussians, "
                                                       "one gradient all-reduce per step"
                                                       + (" (SH slices reduced under the last view, its staged colour "
                                                          "gradients all-gathered)" if world > 1 and args.reduce_early else ""),
               "V_in_view": V, "K_overlaps": K, "K_per_tile_mean": float(counts.mean()),
               "K_per_tile_max": int(counts.max()), "scale_factor": W["scale_factor"],
               "l2_policy": "inputs larger than L2 (708 MB of gaussians per view)", "gaussian_order": "morton" if args.morton else "as generated (random)",
               "emulate_stale_tail": True, "forward_exit_transmittance": 0.0,
               "cuda_graph": use_graph, "cuda_graph_error": graph_state["error"],
               "gradient_sum": ("in-switch reduction through a multicast mapping of the bucket (gs_multimem_all_reduce), "
                                f"inside the step's graph, pipelined with the SH flush in {args.pipeline_chunks} slices"
                                if bucket.reducer is not None else
                                ("ncclAllReduce" if world > 1 else None)),
               "overlap_capacity": graph_state["capacity"] if use_graph else None, "overlap_total_max": overlap_total_max,
               "graph_vs_eager_grad_rel_l2": graph_check,
               "sh": "colours of all views of a step evaluated in one pass over the coefficients, coefficient gradient "
                     "formed once per step" if args.batched_sh else "evaluated per view, coefficient gradient formed once per step"},
    "e2e": {"value": e2e, "unit": "gaussian*pixel/s", "ms_per_step": ms_e2e / args.steps,
            "ms_per_frame": ms_e2e / args.steps / views,
            "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
            "note": "a training step: cameras + target images (8 bit RGB, as a dataset holds them; converted on the device) of the step's views go host -> device from pinned memory "
                    "inside the timed region, the step's loss comes back (read one step late, so the host never drains "
                    "the stream); the gaussians' parameters and their gradient bucket are RESIDENT on the device, as "
                    "they are for a trainer",
            "losses_read_on_host": len(losses_read)},
    "gpu_launches": launches,
    "roofline": {"kernel": "raster_bwd_fast_kernel (gs_raster_bwd)", "bound": "hbm", "achieved": achieved,
                 "peak": peak_gbs, "peak_source": peak_src, "unit": "GB/s",
                 "frac": achieved / peak_gbs if peak_gbs else None, "traffic": traffic,
                 "traffic_source": traffic_src,
                 "algorithmic_bytes": bwd_bytes, "avg_launch_ms": bwd_avg_ms,
                 "note": "instruction bound kernel (SURVEY.md §8d): HBM fraction is low by construction; "
                         "blend_evals_per_s is the informative figure",
                 "blend_evals_per_s": K * 256 / (bwd_avg_ms * 1e-3) if bwd_avg_ms > 0 else None,
                 "issue_roofline": issue},
    "step_tail_ms": {k: round(v, 4) for k, v in phase_ms.items()},
    "single_stream_ms_per_frame": ms_single / stage_steps / views,
    "eager_ms_per_frame": (ms_eager / views) if ms_eager is not None else None,
    "without_stale_tail_ms_per_frame": (ms_no_stale / views) if ms_no_stale is not None else None,
    "stage_ms_note": "entry point times and the roofline come from a second pass with one view stream (kernels timed alone)",
    "stage_ms_per_frame": stage_ms,
    "hbm_stage_rooflines": hbm_stages,
    "clocks": clocks,
  }
  if stock_ms is not None:
    out["stock_api_ms_per_frame"] = stock_ms
    out["stock_api_note"] = ("the reference's call sequence only: render_gaussians(use_sh=True) per view, plain autograd "
                             "accumulation (no sh_colors, no GradientBucket.fused_accumulation); the headline uses those "
                             "two extensions")
  if world > 1:
    dist.destroy_process_group()
  if rank == 0 and world == 1 and not args.no_configs:
    # BASELINE.json's five configurations at full size, fwd+bwd ms per frame through the public API (V, K recorded)
    del gaussians, bucket, params, dev_targets, staged, host_targets
    torch.cuda.empty_cache()
    out["configs"] = run_configs(device)
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    out["cpu_baseline"] = cpu_baseline(W, budget_s=args.cpu_budget)
  if dumped is not None:
    write_outputs(args.dump_outputs, dumped)
  if rank == 0:
    print(json.dumps(out))


DUMP_BYTES = 64_000_000


def sample_outputs(loss, grads, budget=DUMP_BYTES, seed=0):
  """What a caller of the timed step receives, copied to the host as float32 numpy arrays: the step's loss (the sum
  of this rank's view losses) and the gradient of every parameter.  When all gradient rows would take more than
  `budget` bytes, every gradient is cut down to the same rows: a sorted sample of the gaussians drawn from `seed`, so
  that two runs with the same arguments dump the same rows."""
  n = next(iter(grads.values())).shape[0]
  row_bytes = sum(g[0].numel() * 4 for g in grads.values())
  keep = (budget - (1 << 16)) // row_bytes   # 64 KB left for the loss and the .npy headers
  rows = None
  if n > keep:
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
  out = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
  for name, g in grads.items():
    g = g if rows is None else g.index_select(0, rows.to(g.device))
    out[f"grad_{name}"] = g.detach().float().cpu().numpy()
  return out


def write_outputs(directory, arrays):
  import numpy as np
  path = Path(directory)
  path.mkdir(parents=True, exist_ok=True)
  for name, a in arrays.items():
    np.save(path / f"{name}.npy", a)


def run_configs(device, steps=5):
  sys.path.insert(0, str(ROOT / "benchmarks"))
  import configs as cfgs
  res = {}
  for name in ("c1", "c1_graph", "c2", "c3", "c3_graph", "c4", "c5"):
    try:
      maker = cfgs.CONFIGS.get(name) or cfgs.EXTRA[name]
      step = maker(device)
      ms, stages, info = cfgs.timed(step, steps if not name.endswith("_graph") else (50 if name == "c1_graph" else 10))
      res[name] = {"ms_per_frame": round(ms, 3), "what": " ".join(maker.__doc__.split()), **info,
                   "raster_fwd_ms": stages.get("gs_raster_fwd"), "raster_bwd_ms": stages.get("gs_raster_bwd")}
    except Exception as e:   # noqa: BLE001 - report and continue
      res[name] = {"error": f"{type(e).__name__}: {e}"}
    torch.cuda.empty_cache()
  res["note"] = ("single view fwd+bwd, per view SH evaluation; c3 is a synthetic stand-in for the bicycle scene whose only "
                 "published figure is 17.1 ms on an RTX 4090 (reference benchmarks/benchmark-4090.csv:16; target <= 5.7 ms)")
  return res


# ----------------------------------------------------------------------------------------------- CPU legs
def oracle_frame(gaussians, camera, config):
  """One forward + backward frame of the CPU restatement of the reference algorithm (oracle/): C++/OpenMP for the
  projection forward AND backward, SH forward, tile mapping, rasterizer forward / backward; torch (CPU) autograd only
  for the SH coefficient gradient.  Returns (V, K)."""
  import oracle
  from oracle import torch_ref
  g = gaussians
  pts, depth, idx = oracle.project_to_image(g, camera, config)
  feats = torch_ref.evaluate_sh_at(g.feature, g.position.detach(), idx, camera.camera_position)
  ndc = torch_ref.ndc_depth(depth, camera.near_plane, camera.far_plane)
  o2p, ranges = oracle.map_to_tiles(pts, ndc, camera.image_size, config)
  pts.requires_grad_(True)
  raster = oracle.rasterize_with_tiles(pts, feats, o2p, ranges.view(-1, 2), camera.image_size, config)
  raster.image.abs().mean().backward()
  grads, _ = oracle.projection_backward(*g.shape_tensors(), camera.T_camera_world, camera.projection, camera.image_size,
                                        idx, pts.grad, None, blur_cov=config.blur_cov, clamp_margin=config.clamp_margin)
  return int(idx.shape[0]), int(o2p.shape[0])


def cpu_scene(W):
  """The benchmark scene at FULL size on the host (same gaussians, camera and resolution as the GPU arm)."""
  gaussians, cameras, _ = build_scene(W["scene"], W["seed"], 1, W["num_gaussians"], W["image_size"])
  gaussians.feature.requires_grad_(True)
  return gaussians, cameras[0]


def cpu_baseline(W, budget_s=12.0):
  import oracle
  from taichi_gaussian_rasterizer_b200 import RasterConfig
  use_all_host_threads()
  config = RasterConfig(tile_size=W["tile_size"])
  gaussians, camera = cpu_scene(W)
  n = W["num_gaussians"]
  t0 = time.perf_counter()
  frames = 0
  while True:
    gaussians.feature.grad = None
    V, K = oracle_frame(gaussians, camera, config)
    frames += 1
    if time.perf_counter() - t0 > budget_s or frames >= 200:
      break
  dt = (time.perf_counter() - t0) / frames
  w, h = W["image_size"]
  return {"value": n * w * h / dt, "unit": "gaussian*pixel/s", "cores": oracle.num_threads(), "kind": "port",
          "sample": f"{frames} frame(s) of the benchmark scene at FULL size ({n} gaussians, same camera, {w}x{h}, SH3, "
                    f"fwd+bwd): {dt:.2f} s/frame, V={V}, K={K}"}


def use_all_host_threads():
  """torchrun exports OMP_NUM_THREADS=1 for N > 1; the CPU legs are meant to use every host core the process may
  run on, so the thread counts of the OpenMP oracle and of torch are set explicitly."""
  import oracle
  cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
  oracle.set_num_threads(cores)
  torch.set_num_threads(cores)
  return cores


def run_reference(args):
  """The reference's algorithm on the host cores: the Taichi package cannot be installed here (no wheel, no
  network; its rasterizer has no CPU arch anyway, SURVEY.md header), so this arm times oracle/ — the C++/OpenMP
  + torch restatement — with all host threads on the SAME workload at full size; a step is ONE view (the GPU arm's
  step is `views_per_rank` views; the metric is normalised per gaussian and pixel)."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  import oracle
  from taichi_gaussian_rasterizer_b200 import RasterConfig
  use_all_host_threads()
  W, _, scaling = resolve_workload(args)
  config = RasterConfig(tile_size=W["tile_size"])
  gaussians, camera = cpu_scene(W)
  n = W["num_gaussians"]
  w, h = W["image_size"]

  def frame():
    gaussians.feature.grad = None
    return oracle_frame(gaussians, camera, config)

  warmup = min(args.warmup, 1)           # a full-size frame takes seconds: one warm-up frame is enough for a CPU
  for _ in range(warmup):
    frame()
  steps = args.steps
  t0 = time.perf_counter()
  for _ in range(steps):
    V, K = frame()
  dt = (time.perf_counter() - t0) / steps
  value = n * w * h / dt
  sample = (f"each step = 1 frame fwd+bwd of the benchmark scene at FULL size ({n} gaussians, same camera), {w}x{h}, "
            f"SH3; V={V}, K={K}; {steps} timed steps, {dt:.2f} s/frame")
  print(json.dumps({
    "impl": "reference", "metric": "gaussians_px_per_s_fwd_bwd", "value": value, "unit": "gaussian*pixel/s",
    "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "ms_per_frame": dt * 1e3,
    "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    "config": {"workload": workload_name(W),
               "sample": "CPU restatement of the reference algorithm (oracle/, C++/OpenMP) on the full workload, one "
                         "view per step, all host threads"},
    "cpu_baseline": {"value": value, "unit": "gaussian*pixel/s", "cores": oracle.num_threads(), "kind": "port",
                     "sample": sample},
    "e2e": {"value": value, "unit": "gaussian*pixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0}))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
  ap.add_argument("--views-per-rank", type=int, default=8)
  ap.add_argument("--num-gaussians", type=int, default=0)
  ap.add_argument("--image-size", type=int, nargs=2, default=None)
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--per-view-sh", dest="batched_sh", action="store_false",
                  help="evaluate the SH colours per view (evaluate_sh_at) instead of once per step for all views")
  ap.add_argument("--morton", action="store_true", help="store the gaussians in Morton order of their positions")
  ap.add_argument("--cpu-budget", type=float, default=12.0)
  ap.add_argument("--workload", choices=sorted(WORKLOADS), default="bench")
  ap.add_argument("--total-views", type=int, default=0,
                  help="fixed batch split over the ranks (strong scaling), e.g. --workload c5 --total-views 64")
  ap.add_argument("--no-configs", action="store_true", help="skip the per-configuration (c1..c5) timings at N = 1")
  ap.add_argument("--no-stock", action="store_true", help="skip the stock-API (no extensions) timing at N = 1")
  ap.add_argument("--streams", type=int, default=2,
                  help="CUDA streams the views of a step are issued on, round robin (1 = one after another)")
  ap.add_argument("--background-ctas", type=int, default=0,
                  help="N > 1 with reduce_early: CTA limit of the communicator that runs under the last view (0 = default group)")
  ap.add_argument("--stream-priority", type=int, default=-1,
                  help="CUDA priority of the view streams (-1 = high: the rasterizer kernels still launch at the lowest)")
  ap.add_argument("--kernel-variant", type=int, default=0, help="set_raster_options(kernel_variant=): A/B switches")
  ap.add_argument("--symmetric-from", type=int, default=4,
                  help="smallest world size that sums the bucket with the in-switch kernel (below it: ncclAllReduce)")
  ap.add_argument("--pipeline-chunks", type=int, default=4,
                  help="symmetric bucket: slices of the deferred SH flush, each reduced while the next one is formed (1 = off)")
  ap.add_argument("--nccl-bucket", dest="symmetric", action="store_false",
                  help="N > 1: sum the gradient bucket with ncclAllReduce instead of the multimem kernel")
  ap.add_argument("--no-graph", dest="graph", action="store_false",
                  help="issue every step eagerly (kernel launches + two host read-backs per view) instead of replaying it "
                       "from one CUDA graph")
  ap.add_argument("--reduce-early", dest="reduce_early", action="store_true",
                  help="N > 1: reduce the SH slices of the bucket under the last view (measured: the reduction's traffic "
                       "slows that view's rasterizer by what it hides, 21.42 vs 21.22 ms per step on 8 GPUs)")
  ap.add_argument("--no-reduce-early", dest="reduce_early", action="store_false",
                  help="N > 1: one all-reduce of the whole bucket after the last view (the default)")
  ap.set_defaults(reduce_early=False)
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): the loss and "
                       "the gradient of every parameter, cut down to a fixed seeded sample of the gaussians when larger "
                       "than 64 MB in all")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl != "ours":
    ap.error("--dump-outputs writes the outputs of --impl ours")
  if args.impl == "reference":
    run_reference(args)
  else:
    args.warmup = max(args.warmup, 3)
    run_ours(args)


if __name__ == "__main__":
  main()
