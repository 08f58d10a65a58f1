"""Gradient sinks: parameter storage -> buffer that a backward kernel ADDS into, instead of returning a fresh dense
gradient for autograd to accumulate (one read-modify-write pass less per parameter and view, and no dense zero fill
of the culled rows).  Installed by ``distributed.GradientBucket.fused_accumulation()`` around a multi-view batch;
used by the spherical-harmonics backward (feature) and the projection backward (position, log_scaling, rotation,
alpha_logit).  Without a registered sink every operator returns ordinary gradients."""
from typing import Optional

import torch

_sinks = {}


def register_grad_sink(param: torch.Tensor, buffer: torch.Tensor):
  assert buffer.shape == param.shape and buffer.dtype == param.dtype and buffer.is_contiguous()
  _sinks[param.data_ptr()] = buffer


def unregister_grad_sink(param: torch.Tensor):
  _sinks.pop(param.data_ptr(), None)


def grad_sink(param: torch.Tensor) -> Optional[torch.Tensor]:
  return _sinks.get(param.data_ptr())


# ---------------------------------------------------------------------------------------------- deferred SH gradient
def flush_sh_views(sink: torch.Tensor, points: torch.Tensor, staged, camera_positions, overwrite: bool, rows=None):
  """sink (N, K, D) (+)= sum_v staged_v (x) basis(points - camera_v): gs_sh_bwd_flush in chunks of MAX_VIEWS views
  (the first chunk overwrites the rows when ``overwrite``, the others add).  ``rows = (lo, hi)``: only those gaussians
  (row slices of every tensor are contiguous)."""
  import ctypes
  from . import _native as N
  if rows is not None:
    lo, hi = rows
    sink, points, staged = sink[lo:hi], points[lo:hi], [t[lo:hi] for t in staged]
  n, k, d = sink.shape
  if n == 0:
    return
  for c0 in range(0, len(staged), DeferredSH.MAX_VIEWS):
    chunk_s, chunk_c = staged[c0:c0 + DeferredSH.MAX_VIEWS], camera_positions[c0:c0 + DeferredSH.MAX_VIEWS]
    nv = len(chunk_s)
    p = N.GsSHParams(N.dtype_code(sink.dtype), k, d, 1, n, 0, 0 if (overwrite and c0 == 0) else 1, 1)
    arr = ctypes.c_void_p * nv
    N.call("gs_sh_bwd_flush", ctypes.byref(p), ctypes.c_int32(nv), arr(*[t.data_ptr() for t in chunk_s]),
           arr(*[c.data_ptr() for c in chunk_c]), N.ptr(points), N.ptr(sink), N.stream_ptr(sink.device))


class DeferredSH:
  """Pending spherical-harmonics coefficient gradients of a multi-view batch (csrc/point_kernels.cu, "deferred SH
  bwd"): every view stages its masked colour gradient (N, 3) with gs_sh_bwd_stage; ``flush`` adds
  sum_v staged_v (x) basis(position - camera_v) to the sink with ONE pass over the (N, 3, D) rows instead of one
  read-modify-write pass per view.  Flushes by itself after MAX_VIEWS views, unless ``hold`` is set: then the sink is
  not touched until someone takes the pending views (GradientBucket.reduce_early: the sink is inside an all-reduce)."""
  MAX_VIEWS = 16

  def __init__(self, sink: torch.Tensor):
    self.sink = sink
    self.pending = []      # (staged (N,3), camera_pos (3,))
    self.points = None     # (N,3) positions shared by the pending views
    self.overwrite_next = False   # the sink holds nothing yet (mark_clean): the next flush writes instead of adding
    self.hold = False
    self.staging = None    # while held: where the next view stages its colour gradient (peer readable memory)
    self.last_points = None
    self._last_flush = None

  def staging_buffer(self):
    """The buffer the next view should stage into, if the holder asked for a particular one (the one view that may
    follow GradientBucket.reduce_early on the symmetric bucket)."""
    if self.hold and self.staging is not None:
      assert not self.pending, "reduce_early(): exactly one view may follow it (the held staging buffer is taken)"
      return self.staging
    return None

  def mark_clean(self):
    """The caller declares the sink's content void (start of a batch): pending views are dropped and the next flush
    overwrites the rows, so nobody has to zero them (GradientBucket.zero_)."""
    self.pending = []
    self.points = None
    self.overwrite_next = True
    self.hold = False
    self.staging = None

  def add(self, staged: torch.Tensor, camera_pos: torch.Tensor, points: torch.Tensor):
    if self.points is not None and (self.points.data_ptr() != points.data_ptr() or self.points.shape != points.shape):
      assert not self.hold, "positions changed while the SH sink is held by an all-reduce"
      self.flush()
    self.points = points
    self.last_points = points
    # views of a batch may be issued on different CUDA streams (bench.py --streams): remember where this one was staged
    ready = None
    if staged.is_cuda:
      ready = torch.cuda.Event()
      ready.record(torch.cuda.current_stream(staged.device))
    self.pending.append((staged, camera_pos, ready))
    if len(self.pending) >= self.MAX_VIEWS and not self.hold:
      self.flush()

  def take_pending(self):
    """Hand the pending views to the caller (who will flush them itself) and release the hold."""
    self._order_after_producers()
    pending, points = [(p[0], p[1]) for p in self.pending], self.points
    self.pending, self.points, self.hold = [], None, False
    return pending, points

  @staticmethod
  def chunk_bounds(n: int, chunks: int):
    """Row bounds [0, ..., n] of ``flush(chunks=)``: up to ``chunks`` non-empty slices of about equal size, every
    inner bound a multiple of 4 rows.  A slice then starts a multiple of 4 floats into the sink at any row width
    (3 D floats), so the flush kernel keeps the sink's 16 B alignment and a reducer offset stays a multiple of 4 floats."""
    if n <= 0:
      return [0, 0]
    chunks = max(1, min(int(chunks), n))
    bounds = [0]
    for c in range(1, chunks + 1):
      b = min(n, -(-((n * c) // chunks) // 4) * 4)
      if b > bounds[-1]:
        bounds.append(b)
    return bounds

  def flush(self, chunks: int = 1, after_chunk=None):
    """``chunks`` > 1: the rows are flushed in that many slices and ``after_chunk(lo, hi)`` is called after each
    slice's kernel has been enqueued (GradientBucket.all_reduce starts reducing a slice while the next one is formed)."""
    if not self.pending and not self.overwrite_next:
      self.points = None
      return False
    self._order_after_producers()
    bounds = self.chunk_bounds(self.sink.shape[0], chunks)
    for lo, hi in zip(bounds, bounds[1:]):
      if len(self.pending) == 0:   # clean sink, nothing staged: the rows become zeros
        self.sink[lo:hi].zero_()
      else:
        flush_sh_views(self.sink, self.points, [p[0] for p in self.pending], [p[1] for p in self.pending],
                       self.overwrite_next, **({"rows": (lo, hi)} if len(bounds) > 2 else {}))
      if after_chunk is not None:
        after_chunk(lo, hi)
    if self.sink.is_cuda:
      self._last_flush = torch.cuda.Event()
      self._last_flush.record(torch.cuda.current_stream(self.sink.device))
    self.overwrite_next = False
    self.pending = []
    self.points = None
    return True

  def _order_after_producers(self):
    """The flushing stream waits for every stream a pending view was staged on and for the previous flush (two
    flushes read-modify-write the same rows)."""
    if not self.sink.is_cuda:
      return
    cur = torch.cuda.current_stream(self.sink.device)
    for p in self.pending:
      if p[2] is not None:
        cur.wait_event(p[2])
        p[0].record_stream(cur)   # staged on another stream's pool, read here: the allocator must not recycle it early
    if self._last_flush is not None:
      cur.wait_event(self._last_flush)


_deferred = {}


def register_deferred_sh(param: torch.Tensor, sink: torch.Tensor) -> DeferredSH:
  d = DeferredSH(sink)
  _deferred[param.data_ptr()] = d
  return d


def unregister_deferred_sh(param: torch.Tensor):
  d = _deferred.pop(param.data_ptr(), None)
  if d is not None:
    d.flush()


def deferred_sh(param: torch.Tensor) -> Optional[DeferredSH]:
  return _deferred.get(param.data_ptr())


def flush_deferred():
  for d in list(_deferred.values()):
    d.flush()
