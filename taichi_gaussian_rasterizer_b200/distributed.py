"""View-parallel rendering across GPUs (one process per GPU, torch.distributed).

The reference is single process / single GPU (SURVEY.md §2: no collective call sites).  A single view
does not shard (global sort, per tile lists over all gaussians), views are independent: every rank holds
a replica of the gaussians, renders its share of a batch of cameras (rank r takes views r::world),
accumulates dense gradients locally and the ranks sum them ONCE per batch with a single all-reduce over
one flat bucket (NCCL over NVLink on the B200 box, gloo in the CPU tests).  Camera gradients are per
view and stay local.
"""
from contextlib import contextmanager
from typing import Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist


def partition_views(num_views: int, rank: int, world_size: int) -> List[int]:
  """Indices of the views rendered by `rank` (round robin, so any prefix of the batch stays balanced)."""
  return list(range(rank, num_views, world_size))


class GradientBucket:
  """One flat buffer holding the gradients of a fixed set of parameters, views into it installed as
  ``param.grad`` so that autograd accumulates straight into the bucket (no flatten copy before the
  all-reduce)."""

  def __init__(self, params: Sequence[torch.Tensor], symmetric: bool = False, group=None):
    """``symmetric``: allocate the bucket in symmetric memory with an NVSwitch multicast mapping and sum it with
    gs_multimem_all_reduce (the reduction happens inside the switch) instead of ncclAllReduce; collective call (every
    rank of ``group``), falls back to an ordinary allocation when the box or the build cannot do it
    (``self.reducer is None``)."""
    self.params = [p for p in params if p.requires_grad]
    assert len(self.params) > 0
    dtype, device = self.params[0].dtype, self.params[0].device
    sizes = [p.numel() for p in self.params]
    self.reducer = None
    self.flat = None
    self.pipeline_chunks = 4   # symmetric bucket: slices of the SH flush reduced while the next one is formed (1 = off)
    if symmetric and device.type == "cuda" and dtype == torch.float32:
      self.reducer = SymmetricBucketReducer.create(sum(sizes), device, group)
      if self.reducer is not None:
        self.flat = self.reducer.buffer
    if self.flat is None:
      self.flat = torch.zeros((sum(sizes),), dtype=dtype, device=device)
    self._early = None            # state of reduce_early(): (split offset, deferred objects on hold, work handle)
    self.background_group = None  # optional low-CTA communicator for the overlapped reduction (make_background_group)
    self._gather_buffers = {}     # all-gather targets of the last views' staged colour gradients, kept across steps
    off = 0
    for p, n in zip(self.params, sizes):
      p.grad = self.flat[off:off + n].view_as(p)
      off += n

  def zero_(self):
    """Zero the gradients.  Inside ``fused_accumulation()`` the SH coefficient slices are not touched: their deferred
    state is marked clean and the batch's first flush overwrites them (no 4 K D bytes per gaussian of zero fill, no read
    of the rows by that flush).  Every view's SH coefficient gradient reaches those slices through that flush."""
    from . import grad_sinks
    assert self._early is None, "reduce_early() must be followed by all_reduce() before the bucket is zeroed"
    clean = [(p, grad_sinks.deferred_sh(p)) for p in self.params]
    clean = [(p, d) for p, d in clean if d is not None]
    if not clean:
      self.flat.zero_()
      return
    skip = {p.grad.data_ptr() for p, _ in clean}
    for p in self.params:
      if p.grad.data_ptr() not in skip:
        p.grad.zero_()
    for _, d in clean:
      d.mark_clean()

  @contextmanager
  def fused_accumulation(self):
    """Inside this context the spherical-harmonics backward and the projection backward add their gradients straight
    into the bucket (in the kernel) instead of materialising dense tensors for autograd to add: per view that removes
    a read-modify-write pass over every gradient (576 MB of SH + 132 MB of geometry at 3 M gaussians) and the zero
    fill of the culled rows.  Results are the same sums; parameters the kernels cannot serve this way (other
    dtypes, features used without SH) keep the normal autograd accumulation.

    The SH coefficient gradient (N, 3, 1 | 4 | 9 | 16, f32: spherical_harmonics.sh_fast_path) of the batch is formed ONCE, by ``flush()`` (called on exit and by
    ``all_reduce``): each view only stages its masked colour gradient (N, 3) and the flush adds
    sum_v staged_v (x) basis(position - camera_v) — one pass over the coefficient rows per batch (or per 16 views)
    instead of one read-modify-write pass per view (grad_sinks.DeferredSH).  Anything that reads the SH gradient
    inside the context (an optimizer step, say) must call ``flush()`` first."""
    from . import grad_sinks
    from .spherical_harmonics import sh_fast_path
    served = [p for p in self.params if p.is_cuda and p.grad is not None]
    deferred = [p for p in served if sh_fast_path(p)]
    for p in served:
      grad_sinks.register_grad_sink(p, p.grad)
    for p in deferred:
      grad_sinks.register_deferred_sh(p, p.grad)
    try:
      yield self
    finally:
      for p in deferred:
        grad_sinks.unregister_deferred_sh(p)   # flushes
      for p in served:
        grad_sinks.unregister_grad_sink(p)

  def flush(self):
    """Add the pending deferred SH gradients (fused_accumulation()) to the bucket."""
    from . import grad_sinks
    for p in self.params:
      d = grad_sinks.deferred_sh(p)
      if d is not None:
        d.flush()

  @property
  def nbytes(self) -> int:
    return self.flat.numel() * self.flat.element_size()

  # ------------------------------------------------------------------------------------------------ collectives
  def _pending_split(self):
    """(element offset where the deferred SH slices start, the deferred objects) when the bucket is laid out
    [parameters without deferred state | parameters with it] and something is pending; else (None, [])."""
    from . import grad_sinks
    offs, off = {}, 0
    for p in self.params:
      offs[id(p)] = off
      off += p.numel()
    deferred = [(p, grad_sinks.deferred_sh(p)) for p in self.params]
    deferred = [(p, d) for p, d in deferred if d is not None]
    live = [(p, d) for p, d in deferred if d.pending or d.overwrite_next]
    if not live:
      return None, []
    first = min(offs[id(p)] for p, _ in live)
    tail = [p for p in self.params if offs[id(p)] >= first]
    if 0 < first and all(any(q is p for q, _ in live) for p in tail):
      return first, [d for _, d in live]
    return None, []

  def reduce_early(self, group=None):
    """Call when all views of the batch EXCEPT THE LAST ONE of this rank have been back-propagated (every rank must
    call it at the same point; no-op on a single rank).  The deferred SH coefficient gradients of the views so far are
    flushed into the bucket and the SH slices — four fifths of the bucket's bytes — are all-reduced right away, on the
    communicator's stream, UNDER the rendering of the last view.  The last view only stages its (N, 3) colour gradient
    (the deferred state is put on hold, the slices are not touched while they are inside the collective);
    ``all_reduce()`` then all-gathers those small staged gradients and camera centres from all ranks and adds
    sum_ranks staged (x) basis to the reduced rows locally.  All-reduce is linear, so the result is the same sum."""
    active = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if not active or self._early is not None:
      return
    split, deferred = self._pending_split()
    if split is None:
      return
    if self.reducer is not None:
      if split % 4 != 0 or len(deferred) != 1:
        return   # the symmetric path serves one deferred SH parameter at a 16 B aligned offset; else reduce at the end
      d = deferred[0]
      self.reducer.ensure_staging(d.sink.shape[0])
      d.flush()
      d.hold = True
      d.staging = self.reducer.staging()[0]   # the last view stages its colour gradient where the peers can read it
      # the in-switch reduction of the SH slices takes a handful of CTAs (the switch does the adding): it runs on its own
      # stream UNDER the last view, whose issue bound kernels keep the other SMs
      cur = torch.cuda.current_stream(self.flat.device)
      side = self.reducer.stream
      side.wait_stream(cur)
      with torch.cuda.stream(side):
        self.reducer.all_reduce(offset=split, channel=1)
        done = torch.cuda.Event()
        done.record(side)
      self._early = (split, deferred, done)
      return
    for d in deferred:
      d.flush()
      d.hold = True
    # this collective runs UNDER the last view's kernels, which are issue bound and fill every SM: a communicator
    # limited to a few CTAs (background_group) takes few SMs away from them and still has the whole view to finish
    work = dist.all_reduce(self.flat[split:], op=dist.ReduceOp.SUM, group=self.background_group or group, async_op=True)
    self._early = (split, deferred, work)

  def _all_reduce_pipelined(self, split, d):
    """The compute step in front of the collective (the flush that forms the SH coefficient rows, HBM bound) and the
    in-switch reduction (NVLink bound) as a pipeline: the geometry head is reduced while the first slice of rows is
    formed, and every slice is reduced while the next one is formed — on the reducer's stream, joined at the end."""
    red = self.reducer
    cur = torch.cuda.current_stream(self.flat.device)
    side = red.stream
    side.wait_stream(cur)                       # every view's backward has been joined into `cur`
    with torch.cuda.stream(side):
      red.all_reduce(offset=0, count=split, channel=1)
    row = d.sink.shape[1] * d.sink.shape[2]

    def after_chunk(lo, hi):
      formed = torch.cuda.Event()
      formed.record(cur)
      side.wait_event(formed)
      with torch.cuda.stream(side):
        red.all_reduce(offset=split + lo * row, count=(hi - lo) * row, channel=1)

    if not d.flush(chunks=self.pipeline_chunks, after_chunk=after_chunk):
      with torch.cuda.stream(side):             # nothing was pending: the rows are final as they are
        red.all_reduce(offset=split, channel=1)
    cur.wait_stream(side)

  def _finish_early_symmetric(self):
    """After reduce_early() on the symmetric bucket: the geometry head is reduced in the switch, then ONE flush kernel
    adds sum_ranks staged_rank (x) basis(position - camera_rank) to the (already reduced) SH rows, reading every rank's
    staged colour gradient of its last view straight from that rank's memory over NVLink — the all-gather and the
    computation that consumes it are one kernel."""
    from . import grad_sinks
    split, deferred, done = self._early
    self._early = None
    d = deferred[0]
    pending, points = d.take_pending()
    d.staging = None
    red = self.reducer
    cur = torch.cuda.current_stream(self.flat.device)
    own_staged, own_cam = red.staging()
    assert len(pending) <= 1, "reduce_early(): exactly one view may follow it"
    if pending:
      staged, cam = pending[0]
      if staged.data_ptr() != own_staged.data_ptr():
        own_staged.copy_(staged)
      own_cam.copy_(cam.reshape(3))
    else:
      own_staged.zero_()
      points = d.last_points
    cur.wait_event(done)                      # the early reduction of the SH slices (reducer.stream)
    red.all_reduce(offset=0, count=split, channel=0)   # geometry head; its opening barrier also tells every rank that
    #                                                    all staging areas are written
    staged_all, cams_all = zip(*[red.staging(q) for q in range(red.world)])
    grad_sinks.flush_sh_views(d.sink, points, list(staged_all), list(cams_all), overwrite=False)
    red.barrier(channel=2)   # nobody's staging area is overwritten (next step) while a peer still reads it

  def _finish_early(self, group):
    if self.reducer is not None:
      return self._finish_early_symmetric()
    split, deferred, work = self._early
    self._early = None
    world = dist.get_world_size(group)
    gathered = []
    for d in deferred:
      pending, points = d.take_pending()
      if not pending:
        continue
      # this rank's staged colour gradients (P, N, 3) and camera centres (P, 3) -> every rank's (world P, ...)
      local = pending[0][0].unsqueeze(0) if len(pending) == 1 else torch.stack([t for t, _ in pending])   # no copy for one view
      cams = torch.stack([c.reshape(3) for _, c in pending])
      key = (id(d), tuple(local.shape))
      buf = self._gather_buffers.get(key)
      if buf is None:
        buf = self._gather_buffers[key] = (local.new_empty((world * local.shape[0], *local.shape[1:])),
                                           cams.new_empty((world * cams.shape[0], 3)))
      w1 = dist.all_gather_into_tensor(buf[0], local, group=group, async_op=True)
      w2 = dist.all_gather_into_tensor(buf[1], cams, group=group, async_op=True)
      gathered.append((d, points, buf, w1, w2))
    # the geometry head follows the gathers on the communicator's stream and runs while the flush below computes
    head = dist.all_reduce(self.flat[:split], op=dist.ReduceOp.SUM, group=group, async_op=True)
    from . import grad_sinks
    work.wait()
    for d, points, (staged_all, cams_all), w1, w2 in gathered:
      w1.wait()
      w2.wait()
      grad_sinks.flush_sh_views(d.sink, points, list(staged_all.unbind(0)), list(cams_all.unbind(0)), overwrite=False)
    head.wait()

  def all_reduce(self, group=None, async_op: bool = False):
    """Sum the bucket over ranks (no-op without an initialised process group / single rank).  With deferred SH
    gradients pending, the part of the bucket that is already final (the geometry gradients in front of the SH slices)
    is reduced while the flush kernel forms the SH rows, then the SH part follows; after ``reduce_early()`` only the
    geometry head and the last view's staged colour gradients are left to exchange."""
    active = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if not active:
      self.flush()
      return None
    if self._early is not None:
      assert not async_op, "all_reduce(async_op=True) after reduce_early() is not supported"
      self._finish_early(group)
      return None
    split, deferred = (None, []) if async_op else self._pending_split()
    if self.reducer is not None and not async_op:
      if split is not None and split % 4 == 0 and len(deferred) == 1 and self.pipeline_chunks > 1:
        self._all_reduce_pipelined(split, deferred[0])
        return None
      self.flush()
      self.reducer.all_reduce()   # on the current stream: in-switch reduction through the multicast mapping
      return None
    if split is None:
      self.flush()
      return dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
    head = dist.all_reduce(self.flat[:split], op=dist.ReduceOp.SUM, group=group, async_op=True)
    self.flush()
    dist.all_reduce(self.flat[split:], op=dist.ReduceOp.SUM, group=group)
    head.wait()
    return None


class SymmetricBucketReducer:
  """A flat f32 buffer in symmetric memory (torch.distributed._symmetric_memory: every rank's replica mapped into
  every rank's address space, plus ONE multicast address per offset that the NVSwitch resolves to all replicas) and its
  in-place sum over the ranks by csrc/multimem_reduce.cu (gs_multimem_all_reduce: multimem.ld_reduce of the rank's
  slice, multimem.st to all replicas, flag barriers in peer memory on both sides).  The kernel runs on the CURRENT
  stream like any other kernel of the step — no communicator stream, no host-side collective call — and can be
  captured in the step's CUDA graph.  Measured on 8 B200 (benchmarks/allreduce_probe.py, 708 MB): 1.59 ms with 8 CTAs
  against 1.74 ms for ncclAllReduce, bit-identical sums."""

  BLOCKS = 16     # CTAs of the reduction kernel: the switch does the adding, 8 CTAs already keep the links full
  CHANNELS = 4    # independent flag sets (reductions / barriers that may be in flight at the same time)

  def __init__(self, buffer, handle, flags, flags_handle, group, blocks):
    self.buffer, self.handle, self.flags, self.flags_handle, self.group = buffer, handle, flags, flags_handle, group
    self.rank, self.world, self.blocks = dist.get_rank(group), dist.get_world_size(group), blocks
    self.stream = torch.cuda.Stream(device=buffer.device, priority=-1)   # for reductions that overlap compute
    self._staging = None   # (tensor, handle, rows): per rank staging area the peers read (ensure_staging)

  @classmethod
  def create(cls, num_floats: int, device, group=None, blocks: Optional[int] = None):
    """Collective.  None when there is no process group / one rank / no multicast support."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2 \
        or dist.get_backend(group) != "nccl":
      return None
    try:
      import ctypes
      import torch.distributed._symmetric_memory as symm_mem
      from . import _native as N
      pg = group if group is not None else dist.group.WORLD
      world = dist.get_world_size(group)
      blocks = int(blocks or cls.BLOCKS)
      buf = symm_mem.empty(int(num_floats), dtype=torch.float32, device=device)
      handle = symm_mem.rendezvous(buf, pg)
      words = int(N.lib().gs_multimem_all_reduce_flag_words(ctypes.c_int32(world), ctypes.c_int32(blocks),
                                                            ctypes.c_int32(cls.CHANNELS)))
      flags = symm_mem.empty(words, dtype=torch.int32, device=device)
      flags.zero_()
      flags_handle = symm_mem.rendezvous(flags, pg)
      ok = torch.tensor([1 if int(handle.multicast_ptr) != 0 else 0], device=device)
      dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)   # also orders the zero fill before anyone's first flag
      torch.cuda.synchronize(device)
      if int(ok.item()) == 0:
        return None
      buf.zero_()
      return cls(buf, handle, flags, flags_handle, group, blocks)
    except Exception as e:   # noqa: BLE001 - no symmetric memory in this torch / on this box: the caller uses NCCL
      import warnings
      warnings.warn(f"symmetric gradient bucket unavailable ({type(e).__name__}: {e}); falling back to ncclAllReduce")
      return None

  def all_reduce(self, offset: int = 0, count: Optional[int] = None, channel: int = 0):
    """Sum ``buffer[offset : offset + count]`` over the ranks, in place, on the current stream (offset: a multiple of
    four floats).  Every rank must issue the same sequence of calls per channel."""
    import ctypes
    from . import _native as N
    count = self.buffer.numel() - offset if count is None else int(count)
    assert offset % 4 == 0 and 0 <= offset and offset + count <= self.buffer.numel() and 0 <= channel < self.CHANNELS
    N.call("gs_multimem_all_reduce", ctypes.c_void_p(int(self.handle.multicast_ptr) + 4 * int(offset)),
           ctypes.c_int64(count), ctypes.c_int32(self.rank), ctypes.c_int32(self.world),
           ctypes.c_void_p(int(self.flags_handle.buffer_ptrs_dev)), ctypes.c_int32(self.blocks), ctypes.c_int32(channel),
           N.stream_ptr(self.buffer.device))

  def barrier(self, channel: int):
    """The ranks meet on the current stream (gs_cross_rank_barrier): whatever each of them enqueued before is complete
    and visible to its peers afterwards."""
    import ctypes
    from . import _native as N
    N.call("gs_cross_rank_barrier", ctypes.c_int32(self.rank), ctypes.c_int32(self.world),
           ctypes.c_void_p(int(self.flags_handle.buffer_ptrs_dev)), ctypes.c_int32(self.blocks), ctypes.c_int32(channel),
           N.stream_ptr(self.buffer.device))

  def ensure_staging(self, rows: int):
    """Per rank staging area in symmetric memory for one view's masked colour gradient (rows, 3) + camera centre (3,),
    which the peers' flush kernels read straight over NVLink.  Collective on first use (and when ``rows`` changes)."""
    if self._staging is not None and self._staging[2] == rows:
      return
    import torch.distributed._symmetric_memory as symm_mem
    pg = self.group if self.group is not None else dist.group.WORLD
    t = symm_mem.empty(rows * 3 + 4, dtype=torch.float32, device=self.buffer.device)
    t.zero_()
    h = symm_mem.rendezvous(t, pg)
    torch.cuda.synchronize(self.buffer.device)
    dist.barrier(group=self.group)
    self._staging = (t, h, rows)

  def staging(self, rank: Optional[int] = None):
    """(staged (rows, 3), camera centre (3,)) views of ``rank``'s staging area (default: this rank's own)."""
    t, h, rows = self._staging
    if rank is None or rank == self.rank:
      return t[:rows * 3].view(rows, 3), t[rows * 3:rows * 3 + 3]
    return (h.get_buffer(rank, (rows, 3), torch.float32, 0), h.get_buffer(rank, (3,), torch.float32, rows * 3))


def run_views(num_views: int, view_fn, streams: Sequence["torch.cuda.Stream"] = (), before_last_view=None):
  """Run ``view_fn(i)`` — forward + loss + backward of view i, gradients accumulating into a GradientBucket inside
  ``fused_accumulation()`` — for i in range(num_views), issued round robin on ``streams`` (CUDA streams; empty or one
  entry = the current stream, one view after another), and return the sum of the scalars the calls returned.

  Views are independent until their gradients meet in the bucket (atomic adds in the kernels, staged colour gradients
  flushed after the join), so with two streams the backward of view i — enqueued without any host wait — runs while
  the host sits in the two read-backs of view i+1's forward (visible count, overlap total), and the tail of one view's
  kernels is filled by the other's: 2.88 -> 2.67 ms per frame on the bench workload (three streams: 2.70).
  ``before_last_view()`` (optional) is called after all earlier views have been joined and before the last one is
  issued (GradientBucket.reduce_early).  Everything is joined back into the current stream before returning."""
  import torch
  main = torch.cuda.current_stream() if torch.cuda.is_available() and len(streams) > 0 else None
  lanes = list(streams) if len(streams) > 1 else [None]
  totals = [None] * len(lanes)

  def fork():
    for s in lanes:
      if s is not None:
        s.wait_stream(main)

  def join():
    for s in lanes:
      if s is not None:
        main.wait_stream(s)

  fork()
  for i in range(num_views):
    if i == num_views - 1 and before_last_view is not None:
      join()
      before_last_view()
      fork()
    lane = i % len(lanes)
    if lanes[lane] is None:
      value = view_fn(i)
    else:
      with torch.cuda.stream(lanes[lane]):
        value = view_fn(i)
        totals[lane] = value if totals[lane] is None else totals[lane] + value
      continue
    totals[lane] = value if totals[lane] is None else totals[lane] + value
  join()
  parts = [t for t in totals if t is not None]
  return sum(parts[1:], parts[0]) if parts else None


def make_background_group(max_ctas: int = 8):
  """A second NCCL communicator over all ranks whose kernels use at most ``max_ctas`` CTAs: for collectives that are
  meant to run underneath compute kernels (GradientBucket.reduce_early) without taking many SMs from them.  Returns
  None when the backend has no such option (gloo) or no process group is initialised."""
  if not (dist.is_available() and dist.is_initialized()) or dist.get_backend() != "nccl":
    return None
  try:
    opts = dist.ProcessGroupNCCL.Options()
    opts.config.max_ctas = int(max_ctas)
    opts.config.min_ctas = 1
    return dist.new_group(ranks=list(range(dist.get_world_size())), backend="nccl", pg_options=opts)
  except Exception:   # noqa: BLE001 - an older torch / NCCL without communicator configs: use the default group
    return None


def all_reduce_statistics(tensors: Iterable[Optional[torch.Tensor]], group=None):
  """Sum per gaussian statistics (visibility (N,), heuristics (N,2) scattered to dense) over ranks."""
  if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
    return
  for t in tensors:
    if t is not None:
      dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
