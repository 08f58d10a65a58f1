"""Spherical harmonics of degree 0 and 2 (and 1, 3 at odd gaussian counts) on the fast SH paths: the batched forward
(gs_sh_fwd_views), the dense atomic-free backward (sh_bwd_dense_kernel), the deferred gradient of
GradientBucket.fused_accumulation() (gs_sh_bwd_stage + gs_sh_bwd_flush), and render_gaussians(..., overlap_capacity=)
eager and captured in a CUDA graph.  At an odd gaussian count the SH slice of a flat gradient bucket is only 4 B
aligned, which the 4 B-unit kernel variants serve."""
from contextlib import contextmanager, nullcontext

import pytest
import torch

from oracle import torch_ref
from taichi_gaussian_rasterizer_b200 import (CapturedStep, RasterConfig, evaluate_sh_at, evaluate_sh_views,
                                             overlap_capacity_for, render_gaussians)
from taichi_gaussian_rasterizer_b200.distributed import GradientBucket, run_views
from taichi_gaussian_rasterizer_b200.torch_lib.projection import join_rt, quat_to_mat
from util import rel_l2, scene3d

pytestmark = pytest.mark.gpu

NAMES = ("position", "log_scaling", "rotation", "alpha_logit", "feature")


def _nearby_cameras(cam, views):
  cams = [cam]
  for k in range(views - 1):
    q = torch.tensor([0.01 * (k % 5 + 1), -0.02 + 0.003 * k, 0.005, 1.0])
    cams.append(cam.transformed(join_rt(quat_to_mat(q / q.norm()), torch.tensor([0.02, 0.001 * k, -0.01]))))
  return cams


def _offset_copy(t, floats=1):
  """A copy of ``t`` whose storage starts ``floats`` floats into a larger buffer (4 B, not 16 B, aligned)."""
  flat = torch.zeros(t.numel() + floats, dtype=t.dtype, device=t.device)
  out = flat[floats:].view_as(t)
  out.copy_(t)
  assert out.data_ptr() % 16 != 0 and out.is_contiguous()
  return out


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("sh_degree", [0, 1, 2, 3])
def test_batched_views_equal_per_view_evaluation(cuda_device, sh_degree, offset):
  """evaluate_sh_views == evaluate_sh_at for every degree, 18 cameras (two gs_sh_fwd_views calls); offset = 1: the
  batched forward reads coefficients that start 4 B past a 16 B boundary (the 4 B-unit instantiation at degree 1, 3).
  The reference colours always come from the 16 B aligned tensor: gs_sh_fwd reads float4 rows at degree 1, 3."""
  g, cam = scene3d(21, 4001, image_size=(256, 192), scale_factor=0.7, sh_degree=sh_degree, margin=1.0)
  cams = [c.to(device=cuda_device) for c in _nearby_cameras(cam, 18)]
  gd = g.to(device=cuda_device)
  feature = _offset_copy(gd.feature) if offset else gd.feature
  every = torch.arange(feature.shape[0], device=cuda_device)
  colors = evaluate_sh_views(feature, gd.position, [c.camera_position for c in cams])
  assert len(colors) == 18
  worst, identical = 0.0, True
  for c, col in zip(cams, colors):
    ref = evaluate_sh_at(gd.feature, gd.position, every, c.camera_position)
    worst = max(worst, (col - ref).abs().max().item())
    identical = identical and torch.equal(col, ref)
  print(f"degree {sh_degree} offset {offset}: max abs difference {worst:.3g}, bit-identical {identical}")
  assert worst <= 1e-6


def _sh_inputs(seed, n, d, device):
  gen = torch.Generator().manual_seed(seed)
  params = (torch.randn(n, 3, d, generator=gen) * 0.4).to(device)
  points = torch.randn(n, 3, generator=gen).to(device)
  cam = torch.tensor([0.3, -0.2, -4.0]).to(device)
  return params, points, cam, gen


@pytest.mark.parametrize("case", ["visible", "culled", "from_out", "from_out_culled", "offset"])
@pytest.mark.parametrize("d", [1, 4, 9, 16])
def test_dense_backward_every_degree(cuda_device, d, case):
  """The dense SH backward (ascending unique indexes) against float64 autograd through oracle/torch_ref.py and against
  the generic atomic kernel.  visible / culled: with a position and camera gradient (the coefficient rows are gathered),
  mostly visible (culled rows zero-filled in the kernel) or mostly culled (memset first); from_out / from_out_culled:
  coefficient gradient only (the clamp mask comes from the forward output, the rows are never read); offset: as
  visible, then gs_sh_bwd called once more on a copy of the coefficients 4 B past a 16 B boundary (the 4 B-unit
  gather at degree 1, 3; called directly because the forward, gs_sh_fwd, reads float4 rows there)."""
  n = 5003
  params, points, cam, gen = _sh_inputs(7 + d, n, d, cuda_device)
  frac = 0.2 if case.endswith("culled") else 0.8
  idx = torch.nonzero(torch.rand(n, generator=gen) < frac).flatten().to(cuda_device)
  gout = (torch.rand(idx.shape[0], 3, generator=gen) - 0.3).to(cuda_device)
  pose = not case.startswith("from_out")

  def run(sorted_unique):
    p = params.clone().requires_grad_(True)
    x = points.clone().requires_grad_(pose)
    c = cam.clone().requires_grad_(pose)
    out = evaluate_sh_at(p, x, idx, c, indexes_sorted_unique=sorted_unique)
    (out * gout).sum().backward()
    grads = [p.grad.clone()] + ([x.grad.clone(), c.grad.clone()] if pose else [])
    p.grad = None
    return out.detach(), grads

  out_d, g_d = run(True)
  out_g, g_g = run(False)
  assert torch.equal(out_d, out_g)
  p64 = params.detach().cpu().double().requires_grad_(True)
  x64 = points.cpu().double().requires_grad_(pose)
  c64 = cam.cpu().double().requires_grad_(pose)
  (torch_ref.evaluate_sh_at(p64, x64, idx.cpu(), c64) * gout.cpu().double()).sum().backward()
  # degree 0: the colour does not depend on the direction, autograd leaves the position / camera gradient unset
  g64 = [t.grad if t.grad is not None else torch.zeros_like(t) for t in [p64] + ([x64, c64] if pose else [])]
  assert g_d[0].abs().sum() > 0
  # the camera gradient is minus the sum of the position gradients: its error is bounded by the size of the summands
  scales = [None, None, g64[1].abs().sum(0).norm().item()] if pose else [None]
  for a, b, r, scale in zip(g_d, g_g, g64, scales):
    if r.norm() == 0:   # degree 0: the colour does not depend on the direction
      assert a.abs().max().item() < 1e-6 and b.abs().max().item() < 1e-6
      continue
    assert rel_l2(a, b) <= 2e-6, rel_l2(a, b)
    if scale is None:
      assert rel_l2(a, r) <= 1e-5, rel_l2(a, r)
    else:
      assert (a.cpu().double() - r).norm().item() <= 1e-5 * scale, ((a.cpu().double() - r).norm().item(), scale)
  if case == "offset":
    import ctypes
    from taichi_gaussian_rasterizer_b200 import _native as N
    shifted = _offset_copy(params)
    g_off = [torch.empty_like(params), torch.empty_like(points), torch.empty_like(cam)]
    p = N.GsSHParams(N.GS_F32, 3, d, 1, n, idx.shape[0], 0, 0)
    N.call("gs_sh_bwd", ctypes.byref(p), N.ptr(shifted), N.ptr(points), N.ptr(idx), N.ptr(cam), N.ptr(gout),
           N.ptr(g_off[0]), N.ptr(g_off[1]), N.ptr(g_off[2]), N.stream_ptr(cuda_device))
    for a, b in zip(g_off, g_d):
      assert torch.equal(a, b) if b.numel() > 3 else rel_l2(a, b) <= 2e-6
  culled = torch.ones(n, dtype=torch.bool, device=cuda_device)
  culled[idx] = False
  assert g_d[0][culled].abs().max().item() == 0.0


@contextmanager
def _plain_sinks(params):
  from taichi_gaussian_rasterizer_b200.grad_sinks import register_grad_sink, unregister_grad_sink
  for p in params:
    register_grad_sink(p, p.grad)
  try:
    yield
  finally:
    for p in params:
      unregister_grad_sink(p)


@pytest.mark.parametrize("sink", ["deferred", "plain"])
@pytest.mark.parametrize("n,views,sh_degree", [(3000, 19, 0), (3000, 19, 2)] +
                         [(n, 3, d) for n in (3001, 4999) for d in (0, 1, 2, 3)])
def test_fused_accumulation_every_degree(cuda_device, n, views, sh_degree, sink):
  """GradientBucket.fused_accumulation() at every degree equals plain autograd accumulation into the bucket: 19 views
  cross the 16-view auto-flush; at N = 3001, 4999 the SH slice starts 11 N floats into the bucket, 4 B past a 16 B
  boundary (4 B-unit flush).  ``plain``: sinks registered by hand, a one-view flush into the slice per view."""
  cfg = RasterConfig()
  g, cam = scene3d(11 + sh_degree, n, image_size=(256, 192), scale_factor=0.7, sh_degree=sh_degree, margin=0.5)
  cams = [c.to(device=cuda_device) for c in _nearby_cameras(cam, views)]

  def run(fused):
    gd = g.to(device=cuda_device)
    gd.requires_grad_(True)
    params = [getattr(gd, name) for name in NAMES]
    bucket = GradientBucket(params)
    assert (gd.feature.grad.data_ptr() % 16 == 0) == (n % 4 == 0)
    ctx = nullcontext() if not fused else bucket.fused_accumulation() if sink == "deferred" else _plain_sinks(params)
    with ctx:
      bucket.flat.fill_(7.0)
      bucket.zero_()
      for i, c in enumerate(cams):
        render_gaussians(gd, c, cfg, use_sh=True).image.square().mean().backward()
        if fused and i == 1:
          bucket.flush()
    return bucket.flat.clone(), gd.feature.grad.clone()

  flat_a, feat_a = run(False)
  flat_b, feat_b = run(True)
  assert feat_a.abs().sum() > 0
  assert rel_l2(feat_b, feat_a) < 2e-6, rel_l2(feat_b, feat_a)
  assert rel_l2(flat_b, flat_a) < 2e-6, rel_l2(flat_b, flat_a)


def _scene(device, n, sh_degree, seed=3):
  g, cam = scene3d(seed, n, image_size=(320, 240), scale_factor=0.5, sh_degree=sh_degree)
  g = g.to(device=device)
  g.requires_grad_(True)
  return g, cam.to(device=device)


@pytest.mark.parametrize("n", [6000, 6001])
@pytest.mark.parametrize("sh_degree", [0, 2])
def test_static_render_equals_default(cuda_device, sh_degree, n):
  """render_gaussians(use_sh=True, overlap_capacity=) at degree 0 and 2 (counted SH forward, staged backward flushed
  into a fresh gradient): image bit-identical to the default path, gradients within 2e-6."""
  cfg = RasterConfig()
  g, cam = _scene(cuda_device, n, sh_degree)
  torch.manual_seed(1)
  gi = None

  def run(**kw):
    nonlocal gi
    for name in NAMES:
      getattr(g, name).grad = None
    out = render_gaussians(g, cam, cfg, use_sh=True, **kw)
    if gi is None:
      gi = torch.rand_like(out.image) - 0.3
    (out.image * gi).sum().backward()
    return out, {name: getattr(g, name).grad.clone() for name in NAMES}

  ref, g_ref = run()
  out, g_out = run(overlap_capacity=overlap_capacity_for(g, [cam], cfg))
  assert torch.equal(out.image, ref.image) and torch.equal(out.image_weight, ref.image_weight)
  for name in NAMES:
    assert rel_l2(g_out[name], g_ref[name]) < 2e-6, (name, rel_l2(g_out[name], g_ref[name]))


@pytest.mark.parametrize("sh_degree", [0, 2])
def test_captured_bucket_step_equals_plain_autograd(cuda_device, sh_degree):
  """The benchmark's step at degree 0 and 2 with an odd gaussian count (SH slice 4 B aligned): three views on two
  streams, batched colours, deferred SH gradient, captured in one CUDA graph; the replay equals an eager step of plain
  autograd accumulation into the bucket, also after the parameters changed in place."""
  cfg = RasterConfig()
  g, cam0 = _scene(cuda_device, 6001, sh_degree)
  cams = [cam0] + [c.to(device=cuda_device) for c in _nearby_cameras(cam0.to(device="cpu"), 3)[1:]]
  targets = [torch.rand(cam0.image_size[1], cam0.image_size[0], 3, device=cuda_device) for _ in cams]
  params = [getattr(g, name) for name in NAMES]
  bucket = GradientBucket(params)
  assert g.feature.grad.data_ptr() % 16 != 0
  streams = [torch.cuda.Stream(device=cuda_device) for _ in range(2)]
  capacity = overlap_capacity_for(g, cams, cfg)

  def captured_step():
    with bucket.fused_accumulation():
      bucket.zero_()
      colors = evaluate_sh_views(g.feature, g.position, [c.camera_position for c in cams])

      def view(i):
        out = render_gaussians(g, cams[i], cfg, use_sh=True, sh_colors=colors[i], overlap_capacity=capacity)
        loss = torch.nn.functional.l1_loss(out.image, targets[i])
        loss.backward()
        return loss.detach()
      total = run_views(len(cams), view, streams)
      bucket.flush()
    return total

  def plain_step():
    bucket.zero_()
    total = 0.0
    for i, c in enumerate(cams):
      loss = torch.nn.functional.l1_loss(render_gaussians(g, c, cfg, use_sh=True).image, targets[i])
      loss.backward()
      total += loss.item()
    torch.cuda.synchronize()
    return total, bucket.flat.clone()

  ref_loss, ref = plain_step()
  captured = CapturedStep(captured_step, device=cuda_device)
  torch.cuda.synchronize()
  bucket.flat.fill_(7.0)
  loss = captured.replay().item()
  assert rel_l2(bucket.flat, ref) < 2e-6, rel_l2(bucket.flat, ref)
  assert abs(loss - ref_loss) <= 1e-6 * abs(ref_loss)
  with torch.no_grad():
    g.alpha_logit.sub_(0.2)
    g.feature.mul_(0.9)
  loss2 = captured.replay().item()
  replayed = bucket.flat.clone()
  moved_loss, moved = plain_step()
  assert abs(loss2 - moved_loss) <= 1e-6 * abs(moved_loss) and loss2 != ref_loss
  assert rel_l2(replayed, moved) < 2e-6, rel_l2(replayed, moved)
