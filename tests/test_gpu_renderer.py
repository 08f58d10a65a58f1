"""render_gaussians end to end on the GPU against the oracle pipeline (projection -> SH -> tile map ->
rasterize) and torch autograd through the torch restatements for the 3D parameter gradients."""
from contextlib import contextmanager, nullcontext

import pytest
import torch

import oracle
from oracle import torch_ref
from taichi_gaussian_rasterizer_b200 import RasterConfig, Rendering, render_gaussians
from util import GRAD_REL_L2, IMAGE_REL_L2, rel_l2, scene3d

pytestmark = pytest.mark.gpu


def oracle_render(g, cam, cfg, use_sh, render_depth, out):
  """float64 CPU reference pipeline with autograd (taichi_splatting/renderer.py:133-231): torch restatements for
  the per point stages, the C++ oracle for tile mapping and rasterization.  The visible set comes from the f32
  C++ oracle (bit-exact contract with the CUDA projection); the tile map is built by the oracle from the SAME
  packed gaussians / sort depths the CUDA path produced, so both sides blend identical lists."""
  p_orc, d_orc, idx = oracle.projection_forward(*[t.detach() for t in g.shape_tensors()], cam.T_camera_world,
                                                cam.projection, cam.image_size, cam.depth_range, cfg.blur_cov,
                                                cfg.clamp_margin, cfg.alpha_threshold)
  assert torch.equal(out.points_in_view.cpu(), idx), "visible set differs from the oracle"
  assert torch.equal(out.gaussians2d.detach().cpu().view(torch.int32), p_orc.view(torch.int32))
  ndc = torch_ref.ndc_depth(out.point_depth.detach().cpu(), cam.near_plane, cam.far_plane)
  o2p, ranges = oracle.map_to_tiles(out.gaussians2d.detach().cpu(), ndc, cam.image_size, cfg)

  g64 = g.to(dtype=torch.float64).requires_grad_(True)
  cam64 = cam.to(dtype=torch.float64)
  pts_all, depth_all = torch_ref.project_all(*g64.shape_tensors(), cam64.T_camera_world, cam64.projection,
                                             cam.image_size, cfg.blur_cov, cfg.clamp_margin)
  pts, depth = pts_all[idx], depth_all[idx]
  if use_sh:
    feats = torch_ref.evaluate_sh_at(g64.feature, g64.position.detach(), idx, cam64.camera_position)
  else:
    feats = g64.feature[idx]
  if render_depth:
    feats = torch.cat([depth, depth ** 2, feats], dim=1)
  raster = oracle.rasterize_with_tiles(pts, feats, o2p, ranges.view(-1, 2), cam.image_size, cfg)

  # f32 image reference: the f32 oracle rasterizes the very same packed gaussians and lists
  if use_sh:
    f32 = oracle.evaluate_sh_at(g.feature.detach(), g.position.detach(), idx, cam.camera_position)
  else:
    f32 = g.feature.detach()[idx]
  if render_depth:
    f32 = torch.cat([d_orc, d_orc ** 2, f32], dim=1)
  img32, w32, vis32 = oracle.raster_forward(p_orc, f32.contiguous(), o2p, ranges.view(-1, 2), cam.image_size, cfg)
  return raster, idx, o2p, g64, (img32, w32, vis32)


@pytest.mark.parametrize("use_sh,render_depth", [(False, False), (True, False), (True, True), (False, True)])
def test_render_gaussians_vs_oracle(cuda_device, use_sh, render_depth):
  cfg = RasterConfig(compute_visibility=True, compute_point_heuristic=True)
  g, cam = scene3d(3, 6000, image_size=(320, 240), scale_factor=0.5, sh_degree=3 if use_sh else None)
  gd, cd = g.to(device=cuda_device), cam.to(device=cuda_device)
  gd.requires_grad_(True)

  out = render_gaussians(gd, cd, cfg, use_sh=use_sh, render_depth=render_depth)
  ref, idx_ref, o2p_ref, gr, (img32, w32, vis32) = oracle_render(g, cam, cfg, use_sh, render_depth, out)
  assert isinstance(out, Rendering)
  ref_image = ref.image[..., 2:] if render_depth else ref.image
  img32_rgb = img32[..., 2:] if render_depth else img32
  assert rel_l2(out.image, img32_rgb) < IMAGE_REL_L2, rel_l2(out.image, img32_rgb)
  assert rel_l2(out.image_weight, w32) < IMAGE_REL_L2
  assert rel_l2(out.point_visibility, vis32) < GRAD_REL_L2
  assert rel_l2(out.image, ref_image) < 1e-4          # f32 path vs the float64 pipeline
  if render_depth:
    assert out.depth.shape == (240, 320) and out.depth_var.shape == (240, 320)
    d_ref = img32[..., 0] / (w32 + 1e-6)
    assert rel_l2(out.depth, d_ref) < IMAGE_REL_L2
    v_ref = img32[..., 1] / (w32 + 1e-6) - d_ref ** 2
    assert rel_l2(out.depth_var, v_ref) < 1e-3

  torch.manual_seed(1)
  gi = torch.rand_like(ref_image)
  (out.image * gi.to(cuda_device)).sum().backward()
  (ref_image * gi.double()).sum().backward()
  errs = {name: rel_l2(getattr(gd, name).grad, getattr(gr, name).grad)
          for name in ("position", "log_scaling", "rotation", "alpha_logit", "feature")}
  print(errs)
  # raster gradients are pinned at 1e-4 in test_gpu_rasterizer.py; through the f32 projection the scale / rotation
  # terms are ill conditioned for any f32 implementation (see test_projection_f32_grads_within_tolerance)
  assert errs["feature"] < GRAD_REL_L2 and errs["alpha_logit"] < GRAD_REL_L2, errs
  assert errs["position"] < 5e-3 and errs["log_scaling"] < 0.3 and errs["rotation"] < 0.3, errs
  assert out.point_heuristic.shape == (idx_ref.shape[0], 2)
  assert out.split_score.shape == out.prune_cost.shape


def test_median_depth_and_depth16(cuda_device):
  cfg = RasterConfig()
  g, cam = scene3d(5, 4000, image_size=(256, 192), scale_factor=0.5)
  out = render_gaussians(g.to(device=cuda_device), cam.to(device=cuda_device), cfg, render_median_depth=True,
                         use_depth16=True)
  assert out.median_depth.shape == (192, 256)
  assert float(out.median_depth.min()) >= 0
  assert out.ndc_median_depth.shape == (192, 256)


def _nearby_cameras(cam, views):
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import join_rt, quat_to_mat
  cams = [cam]
  for k in range(views - 1):
    q = torch.tensor([0.01 * (k % 5 + 1), -0.02 + 0.003 * k, 0.005, 1.0])
    cams.append(cam.transformed(join_rt(quat_to_mat(q / q.norm()), torch.tensor([0.02, 0.001 * k, -0.01]))))
  return cams


@contextmanager
def _plain_sinks(params):
  """What fused_accumulation() does without the deferred SH state: every backward adds into p.grad by itself."""
  from taichi_gaussian_rasterizer_b200.grad_sinks import register_grad_sink, unregister_grad_sink
  for p in params:
    register_grad_sink(p, p.grad)
  try:
    yield
  finally:
    for p in params:
      unregister_grad_sink(p)


@pytest.mark.parametrize("sink", ["deferred", "plain"])
@pytest.mark.parametrize("n,margin,views,sh_degree", [(5000, 0.0, 3, 3), (5000, 2.0, 3, 3), (3000, 0.5, 19, 1)])
def test_fused_gradient_accumulation_matches_autograd(cuda_device, n, margin, views, sh_degree, sink):
  """GradientBucket.fused_accumulation(): the projection backward adds into the bucket inside the kernel and the SH
  coefficient gradient of the batch is formed once by the deferred flush (per view only the masked colour gradient is
  staged; 19 views cross the 16 view auto-flush).  With ``sink = plain`` the sinks are registered by hand and every
  view's SH gradient is added by a one-view flush.  After the batch the bucket must equal plain autograd accumulation
  (same sums, different rounding order).  Nearly all visible / most gaussians culled / SH degree 1."""
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket
  cfg = RasterConfig()
  g, cam = scene3d(11, n, image_size=(256, 192), scale_factor=0.7, sh_degree=sh_degree, margin=margin)
  cams = [c.to(device=cuda_device) for c in _nearby_cameras(cam, views)]

  def run(fused):
    gd = g.to(device=cuda_device)
    gd.requires_grad_(True)
    params = [gd.position, gd.log_scaling, gd.rotation, gd.alpha_logit, gd.feature]
    bucket = GradientBucket(params)
    if not fused:
      ctx = nullcontext()
    else:
      ctx = bucket.fused_accumulation() if sink == "deferred" else _plain_sinks(params)
    with ctx:
      bucket.flat.fill_(7.0)   # stale content: zero_() inside the context must void it (deferred slices: overwritten
      bucket.zero_()           # by the first flush instead of zero-filled)
      for i, c in enumerate(cams):
        out = render_gaussians(gd, c, cfg, use_sh=True)
        out.image.square().mean().backward()
        if fused and i == 1:
          bucket.flush()   # an early flush (e.g. before an optimizer step) must not lose or double anything
    assert gd.feature.grad.data_ptr() >= bucket.flat.data_ptr()   # still views of the bucket
    return bucket.flat.clone(), gd.feature.grad.clone()

  flat_a, feat_a = run(False)
  flat_b, feat_b = run(True)
  assert feat_a.abs().sum() > 0
  assert rel_l2(feat_b, feat_a) < 2e-6
  assert rel_l2(flat_b, flat_a) < 2e-6


def test_pose_gradient_views_in_fused_accumulation(cuda_device):
  """Views whose SH backward also wants the camera gradient (T_camera_world requires grad) inside
  fused_accumulation(): their coefficient gradient must reach the bucket through the batch's deferred flush like any
  other view's, after zero_() voided stale content, and the pose gradient must be plain autograd's."""
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket
  cfg = RasterConfig()
  g, cam = scene3d(13, 5000, image_size=(256, 192), scale_factor=0.7, sh_degree=3)
  cams_cpu = _nearby_cameras(cam, 3)

  def run(fused):
    gd = g.to(device=cuda_device)
    gd.requires_grad_(True)
    bucket = GradientBucket([gd.position, gd.log_scaling, gd.rotation, gd.alpha_logit, gd.feature])
    cams = [c.to(device=cuda_device) for c in cams_cpu]
    for c in cams:
      c.T_camera_world.requires_grad_(True)
    with bucket.fused_accumulation() if fused else nullcontext():
      bucket.flat.fill_(7.0)
      bucket.zero_()
      for c in cams:
        render_gaussians(gd, c, cfg, use_sh=True).image.square().mean().backward()
    return bucket.flat.clone(), torch.stack([c.T_camera_world.grad for c in cams])

  flat_a, pose_a = run(False)
  flat_b, pose_b = run(True)
  assert flat_a.abs().sum() > 0 and pose_a.abs().sum() > 0
  assert rel_l2(flat_b, flat_a) < 2e-6
  assert rel_l2(pose_b, pose_a) < 2e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_camera_position_kernel(cuda_device, dtype):
  """gs_camera_position == inverse(T_camera_world)[:3, 3] (perspective/params.py:75-78 of the reference), for rigid
  and for general affine view matrices; the differentiable torch path is kept when the pose needs a gradient."""
  from taichi_gaussian_rasterizer_b200.synthetic import random_camera
  torch.manual_seed(3)
  for k in range(4):
    cam = random_camera(image_size=(160, 120)).to(dtype=dtype)
    T = cam.T_camera_world.clone()
    if k % 2:   # not a rotation: sheared / scaled
      T[:3, :3] = T[:3, :3] @ (torch.eye(3, dtype=dtype) + 0.3 * torch.rand(3, 3, dtype=dtype))
    ref = torch.linalg.inv(T.double())[:3, 3]
    camd = cam.to(device=cuda_device)
    camd.T_camera_world = T.to(cuda_device)
    got = camd.camera_position
    assert got.dtype == dtype and got.shape == (3,)
    tol = 2e-5 if dtype == torch.float32 else 1e-12
    assert rel_l2(got.cpu(), ref) < tol
    Tg = T.to(cuda_device).requires_grad_(True)
    camd.T_camera_world = Tg
    pos = camd.camera_position
    assert pos.requires_grad
    assert rel_l2(pos.detach().cpu(), ref) < tol


def test_deferred_sh_clean_bucket_without_views(cuda_device):
  """zero_() inside fused_accumulation() only marks the SH slice clean; leaving the context without a
  single staged view must still leave zeros there."""
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket
  g, _ = scene3d(5, 500, image_size=(64, 48), sh_degree=3)
  gd = g.to(device=cuda_device)
  gd.requires_grad_(True)
  bucket = GradientBucket([gd.position, gd.feature])
  with bucket.fused_accumulation():
    bucket.flat.fill_(3.0)
    bucket.zero_()
  assert float(bucket.flat.abs().max()) == 0.0


@pytest.mark.parametrize("sh_degree,margin", [(3, 0.0), (1, 1.5)])
def test_batched_sh_views_match_per_view(cuda_device, sh_degree, margin):
  """evaluate_sh_views (one pass over the coefficients for all views of a batch) gives evaluate_sh_at's colours, and
  render_gaussians(..., sh_colors=) the same image and the same gradients as the per-view evaluation (18 cameras:
  more than one gs_sh_fwd_views call)."""
  from taichi_gaussian_rasterizer_b200 import evaluate_sh_at, evaluate_sh_views
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import join_rt, quat_to_mat
  cfg = RasterConfig()
  g, cam = scene3d(21, 4000, image_size=(256, 192), scale_factor=0.7, sh_degree=sh_degree, margin=margin)
  cams = [cam]
  for k in range(17):
    q = torch.tensor([0.01 * (k % 4 + 1), -0.02 + 0.004 * k, 0.005, 1.0])
    cams.append(cam.transformed(join_rt(quat_to_mat(q / q.norm()), torch.tensor([0.02, 0.002 * k, -0.01]))))
  cams = [c.to(device=cuda_device) for c in cams]

  gd = g.to(device=cuda_device)
  every = torch.arange(gd.feature.shape[0], device=cuda_device)
  colors = evaluate_sh_views(gd.feature, gd.position, [c.camera_position for c in cams])
  assert len(colors) == 18
  for c, col in zip(cams, colors):
    ref = evaluate_sh_at(gd.feature, gd.position, every, c.camera_position)
    assert col.shape == ref.shape
    assert (col - ref).abs().max().item() < 1e-6

  def run(batched):
    gg = g.to(device=cuda_device)
    gg.requires_grad_(True)
    images = []
    for i in (0, 5, 17):
      out = render_gaussians(gg, cams[i], cfg, use_sh=True, sh_colors=colors[i] if batched else None)
      out.image.square().mean().backward()
      images.append(out.image.detach())
    return images, [gg.feature.grad, gg.position.grad, gg.log_scaling.grad, gg.rotation.grad, gg.alpha_logit.grad]

  img_a, grads_a = run(False)
  img_b, grads_b = run(True)
  for a, b in zip(img_a, img_b):
    assert rel_l2(b, a) < 1e-6
  for a, b in zip(grads_a, grads_b):
    assert rel_l2(b, a) < 1e-5


@pytest.mark.parametrize("count", [0, 1, 4095, 4096, 4097, 20000])
def test_counted_sort_and_depth_order(cuda_device, count):
  """gs_radix_sort_pairs_counted / gs_depth_keys_counted (the count stays on the device; the grid covers the
  capacity): same result as the host-sized calls on the prefix, nothing written past the count, and
  _map_to_tiles(depth_order=...) gives the bit-identical tile map."""
  from taichi_gaussian_rasterizer_b200.cuda_lib import radix_sort_pairs, radix_sort_pairs_counted
  from taichi_gaussian_rasterizer_b200.mapper.tile_mapper import _map_to_tiles, launch_depth_order_counted
  cap = 20000
  gen = torch.Generator().manual_seed(count)
  keys = torch.randint(0, 2 ** 31 - 1, (cap,), dtype=torch.int32, generator=gen).to(cuda_device)
  vals = torch.arange(cap, dtype=torch.int32, device=cuda_device)
  cnt = torch.tensor([count], dtype=torch.int32, device=cuda_device)
  k_ref, v_ref = radix_sort_pairs(keys[:count].contiguous(), vals[:count].contiguous())
  k_out, v_out = radix_sort_pairs_counted(keys, vals, cnt)
  assert torch.equal(k_out[:count], k_ref) and torch.equal(v_out[:count], v_ref)

  cfg = RasterConfig()
  g, cam = scene3d(31, cap, image_size=(320, 240), scale_factor=0.7, sh_degree=None)
  from taichi_gaussian_rasterizer_b200.perspective.projection import project_to_image
  g2d, depths, idx = project_to_image(g.to(device=cuda_device), cam.to(device=cuda_device), cfg)
  v = min(count, g2d.shape[0])
  depth_cap = torch.full((cap, 1), float("nan"), device=cuda_device)
  depth_cap[:v] = depths[:v]
  cntv = torch.tensor([v], dtype=torch.int32, device=cuda_device)
  rng = (cam.near_plane, cam.far_plane)
  order = launch_depth_order_counted(depth_cap, cntv, cam.image_size, cfg, False, rng)
  a = _map_to_tiles(g2d[:v].contiguous(), depths[:v].contiguous(), cam.image_size, cfg, False, ndc_range=rng)
  b = _map_to_tiles(g2d[:v].contiguous(), depths[:v].contiguous(), cam.image_size, cfg, False, ndc_range=rng,
                    depth_order=order[:v])
  assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("n,size,margin", [(1, (17, 13), 0.0), (2, (64, 48), 0.0), (31, (33, 65), 0.3), (33, (640, 360), 0.3),
                                           (1000, (255, 257), 2.0), (50000, (1920, 1080), 0.3), (300, (320, 240), -0.9)])
def test_render_gaussians_equals_stagewise_composition(cuda_device, n, size, margin):
  """render_gaussians (mapper front enqueued with the count on the device, colour kernel before the overlap-total
  read-back, cull masks) against the same pipeline composed from the public stage operators (project_to_image ->
  evaluate_sh_at -> map_to_tiles -> rasterize_with_tiles): identical visible set and tile-dependent outputs, bit for
  bit, on odd image sizes, one or two gaussians, mostly culled and (margin < 0) possibly empty views."""
  from taichi_gaussian_rasterizer_b200 import evaluate_sh_at, map_to_tiles, rasterize_with_tiles
  from taichi_gaussian_rasterizer_b200.perspective.projection import project_to_image
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import ndc_depth
  cfg = RasterConfig()
  g, cam = scene3d(100 + n, n, image_size=size, scale_factor=0.8, sh_degree=3, margin=max(margin, 0.0))
  if margin < 0:   # push most gaussians behind the far plane / out of view
    g.position = g.position + torch.tensor([0.0, 0.0, 1.0]) * 1e4 * (torch.rand(n, 1) < 0.9)
  gd, camd = g.to(device=cuda_device), cam.to(device=cuda_device)
  out = render_gaussians(gd, camd, cfg, use_sh=True)

  g2d, depths, idx = project_to_image(gd, camd, cfg)
  feats = evaluate_sh_at(gd.feature, gd.position, idx, camd.camera_position)
  o2p, ranges = map_to_tiles(g2d, ndc_depth(depths, camd.near_plane, camd.far_plane), camd.image_size, cfg)
  ref = rasterize_with_tiles(g2d, feats, o2p, ranges.view(-1, 2), camd.image_size, cfg)
  assert torch.equal(out.points_in_view, idx)
  assert torch.equal(out.gaussians2d, g2d)
  assert torch.equal(out.image, ref.image)
  assert torch.equal(out.image_weight, ref.image_weight)


def test_views_on_two_streams_accumulate_the_same_gradients(cuda_device):
  """distributed.run_views: the views of a batch issued round robin on two CUDA streams (their gradients meet in the
  flat bucket through atomic adds and the deferred SH flush) give the sums of the one-after-another loop."""
  from taichi_gaussian_rasterizer_b200 import evaluate_sh_views
  from taichi_gaussian_rasterizer_b200.distributed import GradientBucket, run_views
  from taichi_gaussian_rasterizer_b200.torch_lib.projection import join_rt, quat_to_mat
  g, cam = scene3d(11, 40_000, image_size=(400, 300), scale_factor=0.8, sh_degree=3)
  cams = [cam]
  for k in range(5):
    q = torch.tensor([0.01 * (k + 1), -0.02 + 0.004 * k, 0.005, 1.0])
    cams.append(cam.transformed(join_rt(quat_to_mat(q / q.norm()), torch.tensor([0.02, 0.002 * k, -0.01]))))
  cams = [c.to(device=cuda_device) for c in cams]
  cfg = RasterConfig()
  targets = [torch.rand(300, 400, 3, device=cuda_device) for _ in cams]

  def batch(streams):
    gd = g.to(device=cuda_device).requires_grad_(True)
    bucket = GradientBucket([gd.position, gd.log_scaling, gd.rotation, gd.alpha_logit, gd.feature])
    with bucket.fused_accumulation():
      bucket.zero_()
      colors = evaluate_sh_views(gd.feature, gd.position, [c.camera_position for c in cams])

      def one(i):
        loss = torch.nn.functional.l1_loss(render_gaussians(gd, cams[i], cfg, use_sh=True, sh_colors=colors[i]).image,
                                           targets[i])
        loss.backward()
        return loss.detach()
      total = run_views(len(cams), one, streams)
      bucket.all_reduce()
    torch.cuda.synchronize()
    return float(total), bucket.flat.clone()

  loss1, flat1 = batch([])
  loss2, flat2 = batch([torch.cuda.Stream(device=cuda_device) for _ in range(2)])
  loss3, flat3 = batch([torch.cuda.Stream(device=cuda_device) for _ in range(3)])
  assert abs(loss1 - loss2) < 1e-6 and abs(loss1 - loss3) < 1e-6
  assert float(flat1.abs().sum()) > 0
  assert rel_l2(flat2, flat1) < 1e-5 and rel_l2(flat3, flat1) < 1e-5
