"""Autograd operators over the C ABI: the host-side mirror of the reference's
`diff_gaussian_rasterization` wrappers (SURVEY.md section 8b).

  preprocess_gaussians  /root/reference/gaussian_renderer/__init__.py:949-958
  render_gaussians      /root/reference/gaussian_renderer/__init__.py:1271-1282
  get_local2j_ids_bool  /root/reference/gaussian_renderer/workload_division.py:721-744
"""
import ctypes as C
import os

import torch

from . import _lib

BLOCK_X, BLOCK_Y, ONE_DIM_BLOCK_SIZE = 16, 16, 256
LAST_R_TOTAL = 0  # instances binned by the most recent render_gaussians calls (reset by the caller)


# torch.cuda.current_stream() costs ~20 us of Python per call and every operator asks for it: a caller that runs a whole
# step on one stream (pipeline.Trainer.step) pins the handle here for the duration of the step (None = ask torch)
STEP_STREAM = None


def _stream():
    return STEP_STREAM if STEP_STREAM is not None else torch.cuda.current_stream().cuda_stream


def _f32c(t, name):
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (this operator has no CPU path)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    return t.contiguous()


class LazyMs:
    """Elapsed milliseconds between two CUDA events, resolved on first numeric use.

    cuda_args["stats_collector"]["forward_render_time"/"backward_render_time"] must be readable as
    numbers by finish_strategy_final (/root/reference/gaussian_renderer/workload_division.py:953-957).
    Resolving lazily removes two host syncs per camera from the step; set GS_B200_EAGER_TIMING=1 to
    store plain floats instead."""

    __slots__ = ("_s", "_e", "_v")

    def __init__(self, start, end):
        self._s, self._e, self._v = start, end, None

    def value(self):
        if self._v is None:
            self._e.synchronize()
            self._v = float(self._s.elapsed_time(self._e))
            self._s = self._e = None
        return self._v

    def __float__(self):
        return self.value()

    def __add__(self, o):
        return self.value() + float(o)

    __radd__ = __add__

    def __sub__(self, o):
        return self.value() - float(o)

    def __rsub__(self, o):
        return float(o) - self.value()

    def __mul__(self, o):
        return self.value() * float(o)

    __rmul__ = __mul__

    def __truediv__(self, o):
        return self.value() / float(o)

    def __rtruediv__(self, o):
        return float(o) / self.value()

    def __lt__(self, o):
        return self.value() < float(o)

    def __gt__(self, o):
        return self.value() > float(o)

    def __repr__(self):
        return repr(self.value())

    def __format__(self, spec):
        return format(self.value(), spec)


def _timed(collector, key, start, end):
    if collector is None:
        return
    v = LazyMs(start, end)
    collector[key] = v.value() if os.environ.get("GS_B200_EAGER_TIMING") == "1" else v


class _PreprocessGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, scales, rotations, shs, opacities, rs):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        means3D, scales, rotations = _f32c(means3D, "means3D"), _f32c(scales, "scales"), _f32c(rotations, "rotations")
        shs, opacities = _f32c(shs, "shs"), _f32c(opacities, "opacities")
        P = means3D.shape[0]
        if shs.dim() != 3 or shs.shape[1] != 16 or shs.shape[2] != 3:
            raise ValueError(f"shs must be (P,16,3) (scene/gaussian_model.py:122-125), got {tuple(shs.shape)}")
        if tuple(means3D.shape) != (P, 3) or tuple(scales.shape) != (P, 3) or tuple(rotations.shape) != (P, 4) \
                or opacities.numel() != P or shs.shape[0] != P:
            raise ValueError("inconsistent Gaussian parameter shapes")
        dev = means3D.device
        vm, pm, cp = _f32c(rs.viewmatrix, "viewmatrix"), _f32c(rs.projmatrix, "projmatrix"), _f32c(rs.campos, "campos")
        means2D = torch.empty((P, 2), dtype=torch.float32, device=dev)
        depths = torch.empty((P,), dtype=torch.float32, device=dev)
        radii = torch.empty((P,), dtype=torch.int32, device=dev)
        conic_opacity = torch.empty((P, 4), dtype=torch.float32, device=dev)
        rgb = torch.empty((P, 3), dtype=torch.float32, device=dev)
        clamped = torch.empty((P,), dtype=torch.uint8, device=dev)
        _lib.call("gs_preprocess_forward", P, int(rs.sh_degree), means3D.data_ptr(), scales.data_ptr(),
                  float(rs.scale_modifier), rotations.data_ptr(), opacities.data_ptr(), shs.data_ptr(), vm.data_ptr(),
                  pm.data_ptr(), cp.data_ptr(), int(rs.image_width), int(rs.image_height), float(rs.tanfovx),
                  float(rs.tanfovy), means2D.data_ptr(), depths.data_ptr(), radii.data_ptr(), conic_opacity.data_ptr(),
                  rgb.data_ptr(), clamped.data_ptr(), _stream())
        ctx.rs = rs
        ctx.cam = (vm, pm, cp)
        ctx.save_for_backward(means3D, scales, rotations, shs, radii, clamped)
        ctx.mark_non_differentiable(radii, depths)
        return means2D, rgb, conic_opacity, radii, depths

    @staticmethod
    def backward(ctx, g_means2D, g_rgb, g_conic_opacity, _g_radii, _g_depths):
        means3D, scales, rotations, shs, radii, clamped = ctx.saved_tensors
        rs = ctx.rs
        vm, pm, cp = ctx.cam
        P = means3D.shape[0]
        dev = means3D.device

        def z(g, shape):
            return torch.zeros(shape, dtype=torch.float32, device=dev) if g is None else _f32c(g, "grad")

        g_means2D, g_rgb, g_conic_opacity = z(g_means2D, (P, 2)), z(g_rgb, (P, 3)), z(g_conic_opacity, (P, 4))
        d_means3D = torch.empty((P, 3), dtype=torch.float32, device=dev)
        d_scales = torch.empty((P, 3), dtype=torch.float32, device=dev)
        d_rot = torch.empty((P, 4), dtype=torch.float32, device=dev)
        d_opac = torch.empty((P, 1), dtype=torch.float32, device=dev)
        d_shs = torch.empty((P, 16, 3), dtype=torch.float32, device=dev)
        _lib.call("gs_preprocess_backward", P, int(rs.sh_degree), means3D.data_ptr(), scales.data_ptr(),
                  float(rs.scale_modifier), rotations.data_ptr(), shs.data_ptr(), vm.data_ptr(), pm.data_ptr(),
                  cp.data_ptr(), int(rs.image_width), int(rs.image_height), float(rs.tanfovx), float(rs.tanfovy),
                  radii.data_ptr(), clamped.data_ptr(), g_means2D.data_ptr(), g_conic_opacity.data_ptr(),
                  g_rgb.data_ptr(), d_means3D.data_ptr(), d_scales.data_ptr(), d_rot.data_ptr(), d_opac.data_ptr(),
                  d_shs.data_ptr(), _stream())
        return d_means3D, d_scales, d_rot, d_shs, d_opac, None


def preprocess_gaussians(means3D, scales, rotations, shs, opacities, raster_settings, cuda_args=None):
    """-> (means2D (P,2) pixels, rgb (P,3), conic_opacity (P,4), radii (P) int32, depths (P))."""
    return _PreprocessGaussians.apply(means3D, scales, rotations, shs, opacities, raster_settings)


class _PreprocessGaussiansRaw(torch.autograd.Function):
    """preprocess_gaussians with the GaussianModel activations fused in (gs_preprocess_*_raw)."""

    @staticmethod
    def forward(ctx, xyz, f_dc, f_rest, scaling, rotation, opacity, rs):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        xyz, f_dc, f_rest = _f32c(xyz, "_xyz"), _f32c(f_dc, "_features_dc"), _f32c(f_rest, "_features_rest")
        scaling, rotation, opacity = _f32c(scaling, "_scaling"), _f32c(rotation, "_rotation"), _f32c(opacity, "_opacity")
        P = xyz.shape[0]
        if tuple(f_dc.shape) != (P, 1, 3) or tuple(f_rest.shape) != (P, 15, 3):
            raise ValueError("features must be (P,1,3) and (P,15,3) (scene/gaussian_model.py:219-228)")
        if tuple(xyz.shape) != (P, 3) or tuple(scaling.shape) != (P, 3) or tuple(rotation.shape) != (P, 4) \
                or opacity.numel() != P:
            raise ValueError("inconsistent Gaussian parameter shapes")
        dev = xyz.device
        vm, pm, cp = _f32c(rs.viewmatrix, "viewmatrix"), _f32c(rs.projmatrix, "projmatrix"), _f32c(rs.campos, "campos")
        means2D = torch.empty((P, 2), dtype=torch.float32, device=dev)
        depths = torch.empty((P,), dtype=torch.float32, device=dev)
        radii = torch.empty((P,), dtype=torch.int32, device=dev)
        conic_opacity = torch.empty((P, 4), dtype=torch.float32, device=dev)
        rgb = torch.empty((P, 3), dtype=torch.float32, device=dev)
        clamped = torch.empty((P,), dtype=torch.uint8, device=dev)
        _lib.call("gs_preprocess_forward_raw", P, int(rs.sh_degree), xyz.data_ptr(), f_dc.data_ptr(), f_rest.data_ptr(),
                  scaling.data_ptr(), float(rs.scale_modifier), rotation.data_ptr(), opacity.data_ptr(), vm.data_ptr(),
                  pm.data_ptr(), cp.data_ptr(), int(rs.image_width), int(rs.image_height), float(rs.tanfovx),
                  float(rs.tanfovy), means2D.data_ptr(), depths.data_ptr(), radii.data_ptr(), conic_opacity.data_ptr(),
                  rgb.data_ptr(), clamped.data_ptr(), _stream())
        ctx.rs = rs
        ctx.cam = (vm, pm, cp)
        ctx.save_for_backward(xyz, f_dc, f_rest, scaling, rotation, opacity, radii, clamped)
        ctx.mark_non_differentiable(radii, depths)
        return means2D, rgb, conic_opacity, radii, depths

    @staticmethod
    def backward(ctx, g_means2D, g_rgb, g_conic_opacity, _g_radii, _g_depths):
        xyz, f_dc, f_rest, scaling, rotation, opacity, radii, clamped = ctx.saved_tensors
        rs = ctx.rs
        vm, pm, cp = ctx.cam
        P = xyz.shape[0]
        dev = xyz.device

        def z(g, shape):
            return torch.zeros(shape, dtype=torch.float32, device=dev) if g is None else _f32c(g, "grad")

        g_means2D, g_rgb, g_conic_opacity = z(g_means2D, (P, 2)), z(g_rgb, (P, 3)), z(g_conic_opacity, (P, 4))
        d = [torch.empty_like(t) for t in (xyz, f_dc, f_rest, scaling, rotation, opacity)]
        _lib.call("gs_preprocess_backward_raw", P, int(rs.sh_degree), xyz.data_ptr(), f_dc.data_ptr(), f_rest.data_ptr(),
                  scaling.data_ptr(), float(rs.scale_modifier), rotation.data_ptr(), opacity.data_ptr(), vm.data_ptr(),
                  pm.data_ptr(), cp.data_ptr(), int(rs.image_width), int(rs.image_height), float(rs.tanfovx),
                  float(rs.tanfovy), radii.data_ptr(), clamped.data_ptr(), g_means2D.data_ptr(),
                  g_conic_opacity.data_ptr(), g_rgb.data_ptr(), d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(),
                  d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(), _stream())
        return d[0], d[1], d[2], d[3], d[4], d[5], None


def preprocess_gaussians_raw(xyz, features_dc, features_rest, scaling, rotation, opacity, raster_settings):
    """Same outputs as preprocess_gaussians, from the six RAW GaussianModel parameters
    (scene/gaussian_model.py:219-228); the activations of :109-129 run inside the kernel."""
    return _PreprocessGaussiansRaw.apply(xyz, features_dc, features_rest, scaling, rotation, opacity, raster_settings)


def _tiles(rs):
    return (int(rs.image_height) + BLOCK_Y - 1) // BLOCK_Y, (int(rs.image_width) + BLOCK_X - 1) // BLOCK_X


def _seg_workspace(R, num_tiles, dev, needed):
    """Segment workspace linking a render forward to its backward (gs_render_seg_bytes); None for forward-only calls."""
    if not needed or R == 0:
        return None, 0
    nb = _lib.query("gs_render_seg_bytes", R, num_tiles)
    return torch.empty((nb,), dtype=torch.uint8, device=dev), nb


# Instance-count hints: the render reads its instance count R back from the device (the operator's one host sync, as in
# the reference, which sizes its buffers from num_rendered).  Behind that sync the GPU is idle until the next launch, so
# everything the launch needs is allocated BEFORE the sync from the previous call's R of the same shape (+8 %); only when
# the hint is missing or too small are the buffers allocated after the read-back.
_R_HINT = {}


class _InstanceBuffers:
    __slots__ = ("cap", "tiles", "ids", "sort_temp", "sb", "seg", "segb")

    def __init__(self, cap, num_tiles, dev, needs_grad):
        self.cap = _q(cap)
        self.tiles = torch.empty((2, self.cap), dtype=torch.int32, device=dev)
        self.ids = torch.empty((2, self.cap), dtype=torch.int32, device=dev)
        self.sb = _lib.query("gs_render_sort_temp_bytes", self.cap)
        self.sort_temp = torch.empty((self.sb,), dtype=torch.uint8, device=dev)
        self.seg, self.segb = _seg_workspace(self.cap, num_tiles, dev, needs_grad)

    def row(self, t, r):
        return t.data_ptr() + 4 * self.cap * r


def _instance_buffers_before_sync(key, num_tiles, dev, needs_grad):
    est = _R_HINT.get(key)
    return None if est is None else _InstanceBuffers(est + est // 12 + 4096, num_tiles, dev, needs_grad)


def _instance_buffers_after_sync(key, pre, R, num_tiles, dev, needs_grad):
    _R_HINT[key] = R
    if pre is not None and R <= pre.cap and (R > 0 or pre.seg is None):
        return pre
    return _InstanceBuffers(R, num_tiles, dev, needs_grad)


def _q(n):
    """Buffer sizes that follow a data-dependent count (received splats, instances) are rounded up to 1/16 steps of their
    leading power of two: when the strips of a view move, the counts change a little every step, and exact sizes would
    hand the caching allocator a new size -- eventually a cudaMalloc and a device synchronisation -- every few steps."""
    n = max(int(n), 1)
    q = 1 << max(10, n.bit_length() - 5)
    return (n + q - 1) // q * q


def _grad_block(P, dev):
    """dL/dmeans2D (P,2), dL/dconic_opacity (P,4), dL/drgb (P,3) as consecutive blocks of ONE allocation: the backward
    zeroes them with one memset instead of three (it accumulates into them with RED.ADD)."""
    buf = torch.empty((9 * _q(P),), dtype=torch.float32, device=dev)   # conic first: its rows are read as float4
    return buf[4 * P:6 * P].view(P, 2), buf[:4 * P].view(P, 4), buf[6 * P:9 * P].view(P, 3)


class _RenderGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means2D, conic_opacity, rgb, depths, radii, compute_locally, rs, collector):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        means2D, conic_opacity, rgb = _f32c(means2D, "means2D"), _f32c(conic_opacity, "conic_opacity"), _f32c(rgb, "rgb")
        depths = _f32c(depths, "depths")
        if radii.dtype != torch.int32:
            radii = radii.to(torch.int32)
        radii = radii.contiguous()
        P = means2D.shape[0]
        H, W = int(rs.image_height), int(rs.image_width)
        ty, tx = _tiles(rs)
        T = ty * tx
        dev = means2D.device
        if compute_locally is None:
            cl = torch.ones((T,), dtype=torch.uint8, device=dev)
        else:
            if compute_locally.numel() != T:
                raise ValueError(f"compute_locally must have {ty}x{tx} entries, got {tuple(compute_locally.shape)}")
            cl = compute_locally.contiguous()
            cl = cl.view(torch.uint8) if cl.dtype == torch.bool else cl.to(torch.uint8)
        bg = _f32c(rs.bg, "bg")
        s = _stream()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        Pq = _q(P)
        offsets = torch.empty((Pq,), dtype=torch.int32, device=dev)
        order = torch.empty((Pq,), dtype=torch.int32, device=dev)
        rec = torch.empty((Pq, 12), dtype=torch.float32, device=dev)
        tb = _lib.query("gs_render_count_temp_bytes", Pq)
        temp = torch.empty((tb,), dtype=torch.uint8, device=dev)
        ranges = torch.empty((T, 2), dtype=torch.int32, device=dev)
        image = torch.empty((3, H, W), dtype=torch.float32, device=dev)
        final_T = torch.empty((H, W), dtype=torch.float32, device=dev)
        n_contrib = torch.empty((H, W), dtype=torch.int32, device=dev)
        stats = torch.empty((3,), dtype=torch.int64, device=dev)
        needs_grad = means2D.requires_grad or conic_opacity.requires_grad or rgb.requires_grad
        R = C.c_int64(0)
        ticket = C.c_void_p()
        _lib.call("gs_render_count_launch", 1, None, P, H, W, means2D.data_ptr(), conic_opacity.data_ptr(), rgb.data_ptr(),
                  depths.data_ptr(), radii.data_ptr(), cl.data_ptr(), order.data_ptr(), offsets.data_ptr(),
                  rec.data_ptr(), temp.data_ptr(), tb, C.byref(ticket), s)
        key = (1, H, W, needs_grad)          # not P: the splat count of a strip varies from step to step, R follows it smoothly
        pre = _instance_buffers_before_sync(key, T, dev, needs_grad)    # host work while the count / sort / scan run
        _lib.call("gs_render_count_read", ticket, C.byref(R), s)   # the operator's one host sync
        R = int(R.value)
        global LAST_R_TOTAL
        LAST_R_TOTAL += R
        ib = _instance_buffers_after_sync(key, pre, R, T, dev, needs_grad)
        seg = ib.seg if R > 0 else None
        _lib.call("gs_render_forward", P, R, H, W, means2D.data_ptr(), radii.data_ptr(), cl.data_ptr(),
                  order.data_ptr(), offsets.data_ptr(), rec.data_ptr(), bg.data_ptr(), ib.row(ib.tiles, 0),
                  ib.row(ib.ids, 0), ib.row(ib.tiles, 1), ib.row(ib.ids, 1), ib.sort_temp.data_ptr(), ib.sb, ranges.data_ptr(),
                  image.data_ptr(), final_T.data_ptr(), n_contrib.data_ptr(), stats.data_ptr(), _lib.ptr(seg),
                  ib.segb if seg is not None else 0, s)
        ev1.record()
        _timed(collector, "forward_render_time", ev0, ev1)
        ids_sorted = ib.ids[1]    # a view: the (tile, id) scratch stays alive until the backward has run (16 B / instance)
        ctx.rs, ctx.R, ctx.P, ctx.collector, ctx.seg = rs, R, P, collector, seg
        ctx.save_for_backward(rec, bg, cl, ranges, ids_sorted, final_T, n_contrib)
        n_render, n_consider, n_contrib_sum = stats[0], stats[1], stats[2]
        ctx.mark_non_differentiable(n_render, n_consider, n_contrib_sum)
        return image, n_render, n_consider, n_contrib_sum

    @staticmethod
    def backward(ctx, g_image, *_unused):
        rec, bg, cl, ranges, ids_sorted, final_T, n_contrib = ctx.saved_tensors
        rs, R, P = ctx.rs, ctx.R, ctx.P
        H, W = int(rs.image_height), int(rs.image_width)
        dev = rec.device
        g_image = torch.zeros((3, H, W), dtype=torch.float32, device=dev) if g_image is None else _f32c(g_image, "grad")
        d_means2D, d_conic, d_rgb = _grad_block(P, dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        seg = ctx.seg
        _lib.call("gs_render_backward", P, R, H, W, rec.data_ptr(), bg.data_ptr(), cl.data_ptr(), ranges.data_ptr(),
                  ids_sorted.data_ptr(), final_T.data_ptr(), n_contrib.data_ptr(), g_image.data_ptr(),
                  _lib.ptr(seg), 0 if seg is None else seg.numel(),
                  d_means2D.data_ptr(), d_conic.data_ptr(), d_rgb.data_ptr(), _stream())
        ctx.seg = None
        ev1.record()
        _timed(ctx.collector, "backward_render_time", ev0, ev1)
        return d_means2D, d_conic, d_rgb, None, None, None, None, None


def render_gaussians(means2D, conic_opacity, rgb, depths, radii, compute_locally, raster_settings, cuda_args=None,
                     extended_compute_locally=None):
    """-> (image (3,H,W) with non-local tiles exactly 0, n_render, n_consider, n_contrib).

    extended_compute_locally: the live path passes None (workload_division.py:802-803); the legacy render()
    (gaussian_renderer/__init__.py:458-507) passes the local tile region dilated by one tile
    (workload_division.py:142-156, 435-448).  What the fork's CUDA code did with it is not observable (its source is an
    absent submodule) and every in-tree consumer of the result requires the image to be exactly zero outside
    compute_locally (loss_distribution.py:1875), so the mask is validated -- a (TILE_Y, TILE_X) boolean mask that covers
    compute_locally -- and the blend stays confined to compute_locally."""
    if extended_compute_locally is not None:
        ty, tx = _tiles(raster_settings)
        if extended_compute_locally.numel() != ty * tx:
            raise ValueError(f"extended_compute_locally must have {ty}x{tx} entries, got {tuple(extended_compute_locally.shape)}")
        if compute_locally is not None and bool((compute_locally.reshape(-1).bool() & ~extended_compute_locally.reshape(-1).bool()).any()):
            raise ValueError("extended_compute_locally must cover compute_locally")
    collector = None
    if isinstance(cuda_args, dict):
        collector = cuda_args.setdefault("stats_collector", {})
    return _RenderGaussians.apply(means2D, conic_opacity, rgb, depths, radii, compute_locally, raster_settings, collector)


MAX_VIEWS = 64   # GS_MAX_VIEWS


def _i32_array(vals):
    return (C.c_int32 * len(vals))(*[int(v) for v in vals])


class _RenderGaussiansBatched(torch.autograd.Function):
    """render_gaussians for the B cameras of a batch in ONE pass (gs_render_*_batched): the splats of all cameras
    concatenated (camera k = rows [view_start[k], view_start[k+1])), masks (B,T), images (B,3,H,W)."""

    @staticmethod
    def forward(ctx, means2D, conic_opacity, rgb, depths, radii, compute_locally, view_start, rs, collector):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        means2D, conic_opacity, rgb = _f32c(means2D, "means2D"), _f32c(conic_opacity, "conic_opacity"), _f32c(rgb, "rgb")
        depths = _f32c(depths, "depths")
        if radii.dtype != torch.int32:
            radii = radii.to(torch.int32)
        radii = radii.contiguous()
        B = len(view_start) - 1
        P = int(view_start[B])
        if not 1 <= B <= MAX_VIEWS:
            raise ValueError(f"1..{MAX_VIEWS} views per batched render, got {B}")
        if means2D.shape[0] != P:
            raise ValueError(f"view_start ends at {P} but {means2D.shape[0]} splats were passed")
        H, W = int(rs.image_height), int(rs.image_width)
        ty, tx = _tiles(rs)
        T = ty * tx
        dev = means2D.device
        if compute_locally is None:
            cl = torch.ones((B * T,), dtype=torch.uint8, device=dev)
        else:
            if compute_locally.numel() != B * T:
                raise ValueError(f"compute_locally must have {B}x{ty}x{tx} entries, got {tuple(compute_locally.shape)}")
            cl = compute_locally.contiguous()
            cl = cl.view(torch.uint8) if cl.dtype == torch.bool else cl.to(torch.uint8)
        bg = _f32c(rs.bg, "bg")
        s = _stream()
        vs = _i32_array(view_start)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        Pq = _q(P)
        offsets = torch.empty((Pq,), dtype=torch.int32, device=dev)
        order = torch.empty((Pq,), dtype=torch.int32, device=dev)
        rec = torch.empty((Pq, 12), dtype=torch.float32, device=dev)
        tb = _lib.query("gs_render_count_temp_bytes", Pq)
        temp = torch.empty((tb,), dtype=torch.uint8, device=dev)
        ranges = torch.empty((B * T, 2), dtype=torch.int32, device=dev)
        image = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
        final_T = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        n_contrib = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        stats = torch.empty((B, 3), dtype=torch.int64, device=dev)
        needs_grad = means2D.requires_grad or conic_opacity.requires_grad or rgb.requires_grad
        R = C.c_int64(0)
        ticket = C.c_void_p()
        _lib.call("gs_render_count_launch", B, vs, P, H, W, means2D.data_ptr(), conic_opacity.data_ptr(), rgb.data_ptr(),
                  depths.data_ptr(), radii.data_ptr(), cl.data_ptr(), order.data_ptr(), offsets.data_ptr(),
                  rec.data_ptr(), temp.data_ptr(), tb, C.byref(ticket), s)
        key = (B, H, W, needs_grad)
        pre = _instance_buffers_before_sync(key, B * T, dev, needs_grad)   # host work while the count / sort / scan run
        _lib.call("gs_render_count_read", ticket, C.byref(R), s)    # the operator's one host sync
        R = int(R.value)
        global LAST_R_TOTAL
        LAST_R_TOTAL += R
        ib = _instance_buffers_after_sync(key, pre, R, B * T, dev, needs_grad)
        seg = ib.seg if R > 0 else None
        _lib.call("gs_render_forward_batched", B, vs, R, H, W, means2D.data_ptr(), radii.data_ptr(), cl.data_ptr(),
                  order.data_ptr(), offsets.data_ptr(), rec.data_ptr(), bg.data_ptr(), ib.row(ib.tiles, 0),
                  ib.row(ib.ids, 0), ib.row(ib.tiles, 1), ib.row(ib.ids, 1), ib.sort_temp.data_ptr(), ib.sb, ranges.data_ptr(),
                  image.data_ptr(), final_T.data_ptr(), n_contrib.data_ptr(), stats.data_ptr(), _lib.ptr(seg),
                  ib.segb if seg is not None else 0, s)
        ev1.record()
        _timed(collector, "forward_render_time", ev0, ev1)
        ids_sorted = ib.ids[1]    # a view: the (tile, id) scratch stays alive until the backward has run (16 B / instance)
        ctx.rs, ctx.R, ctx.P, ctx.B, ctx.collector, ctx.seg = rs, R, P, B, collector, seg
        ctx.save_for_backward(rec, bg, cl, ranges, ids_sorted, final_T, n_contrib)
        ctx.mark_non_differentiable(stats)
        return image, stats

    @staticmethod
    def backward(ctx, g_image, _g_stats):
        rec, bg, cl, ranges, ids_sorted, final_T, n_contrib = ctx.saved_tensors
        rs, R, P, B = ctx.rs, ctx.R, ctx.P, ctx.B
        H, W = int(rs.image_height), int(rs.image_width)
        dev = rec.device
        g_image = torch.zeros((B, 3, H, W), dtype=torch.float32, device=dev) if g_image is None else _f32c(g_image, "grad")
        d_means2D, d_conic, d_rgb = _grad_block(P, dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        seg = ctx.seg
        _lib.call("gs_render_backward_batched", B, P, R, H, W, rec.data_ptr(), bg.data_ptr(), cl.data_ptr(),
                  ranges.data_ptr(), ids_sorted.data_ptr(), final_T.data_ptr(), n_contrib.data_ptr(), g_image.data_ptr(),
                  _lib.ptr(seg), 0 if seg is None else seg.numel(),
                  d_means2D.data_ptr(), d_conic.data_ptr(), d_rgb.data_ptr(), _stream())
        ctx.seg = None
        ev1.record()
        _timed(ctx.collector, "backward_render_time", ev0, ev1)
        return d_means2D, d_conic, d_rgb, None, None, None, None, None, None


def render_gaussians_batched(means2D, conic_opacity, rgb, depths, radii, compute_locally, view_start, raster_settings,
                             cuda_args=None):
    """All B cameras of a batch in one pass.  means2D (N,2), conic_opacity (N,4), rgb (N,3), depths (N), radii (N):
    the splats of the B cameras concatenated, camera k = rows [view_start[k], view_start[k+1]) (len(view_start) = B+1);
    compute_locally (B, TILE_Y*TILE_X) (None = everything local); the cameras share the image size and background of
    `raster_settings` (their view / projection matrices were consumed by the preprocess).
    -> (images (B,3,H,W) with non-local tiles exactly 0, stats (B,3) int64 = n_render / n_consider / n_contrib)."""
    collector = None
    if isinstance(cuda_args, dict):
        collector = cuda_args.setdefault("stats_collector", {})
    return _RenderGaussiansBatched.apply(means2D, conic_opacity, rgb, depths, radii, compute_locally,
                                         [int(v) for v in view_start], raster_settings, collector)


class _FusedL1SSIMBatched(torch.autograd.Function):
    @staticmethod
    def forward(ctx, images, gts, rows4):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        images = _f32c(images, "images")
        B, _, H, W = images.shape
        if len(gts) != B or len(rows4) != B:
            raise ValueError("one ground-truth strip and one (row0,row1,count_row0,count_row1) per view")
        keep = []
        for k, (gt, r) in enumerate(zip(gts, rows4)):
            rows = int(r[1]) - int(r[0])
            if rows == 0:
                keep.append(None)
                continue
            if gt is None or gt.dtype != torch.uint8 or not gt.is_cuda:
                raise TypeError("gt strips must be CUDA uint8 tensors (3, rows, W)")
            gt = gt.contiguous()
            if tuple(gt.shape) != (3, rows, W):
                raise ValueError(f"gt strip {k} must be (3,{rows},{W}), got {tuple(gt.shape)}")
            keep.append(gt)
        flat = _i32_array([int(v) for r in rows4 for v in r])
        gptr = (C.c_void_p * B)(*[None if g is None else g.data_ptr() for g in keep])
        tb = _lib.query("gs_loss_temp_bytes_batched", B, flat, W)
        temp = torch.empty((tb,), dtype=torch.uint8, device=images.device)
        out = torch.empty((B, 2), dtype=torch.float32, device=images.device)
        _lib.call("gs_loss_forward_batched", B, H, W, flat, images.data_ptr(), gptr, out.data_ptr(), temp.data_ptr(), tb,
                  _stream())
        ctx.rows4, ctx.gts = flat, keep
        ctx.save_for_backward(images, temp)
        return out

    @staticmethod
    def backward(ctx, g_out):
        images, temp = ctx.saved_tensors
        B, _, H, W = images.shape
        if g_out is None:
            return None, None, None
        g_l1, g_ssim = g_out[:, 0].to(torch.float32).contiguous(), g_out[:, 1].to(torch.float32).contiguous()
        d_images = torch.empty_like(images)
        gptr = (C.c_void_p * B)(*[None if g is None else g.data_ptr() for g in ctx.gts])
        _lib.call("gs_loss_backward_batched", B, H, W, ctx.rows4, images.data_ptr(), gptr, temp.data_ptr(),
                  g_l1.data_ptr(), g_ssim.data_ptr(), d_images.data_ptr(), _stream())
        return d_images, None, None


def fused_l1_ssim_batched(images, gts_u8, rows4):
    """The strip losses of the B cameras of a batch in one launch.  images (B,3,H,W); gts_u8: list of B CUDA uint8
    strips (3,rows,W) (None where rows == 0); rows4: B tuples (row0, row1, count_row0, count_row1).
    -> (B,2) = (Ll1, ssim_loss) per camera, both normalised by 3*H*W; zeros for cameras without rows."""
    return _FusedL1SSIMBatched.apply(images, list(gts_u8), [tuple(int(v) for v in r) for r in rows4])


def image_metrics_batched(images, gts_u8, rows4, saved=False):
    """Held-out image metrics of B views in one launch (gs_metrics_batched); no autograd.
    images (B,3,H,W) float32 CUDA; gts_u8: list of B CUDA uint8 windows (3, row1-row0, W) (None where row1 == row0);
    rows4: B tuples (row0, row1, count_row0, count_row1), as for fused_l1_ssim_batched.  saved=False evaluates
    clamp(image, 0, 1) (train_internal.py:471-478); saved=True the image after the 8-bit PNG round trip of
    render.py:127-138 -> metrics.py:26-36.
    -> (B,3,3) float64 on the device: [v][0][c] = sum |x-y|, [v][1][c] = sum (x-y)^2, [v][2][c] = sum ssim_map, over the
    counted rows of channel c."""
    if not isinstance(images, torch.Tensor) or images.dim() != 4 or images.shape[1] != 3:
        raise ValueError(f"images must be a (B,3,H,W) tensor, got {getattr(images, 'shape', type(images))}")
    images = _f32c(images, "images")
    B, _, H, W = images.shape
    gts_u8, rows4 = list(gts_u8), [tuple(int(v) for v in r) for r in rows4]
    if not 1 <= B <= MAX_VIEWS:
        raise ValueError(f"1..{MAX_VIEWS} views per call, got {B}")
    if len(gts_u8) != B or len(rows4) != B or any(len(r) != 4 for r in rows4):
        raise ValueError("one ground-truth window and one (row0,row1,count_row0,count_row1) per view")
    keep = []
    for k, (gt, (r0, r1, c0, c1)) in enumerate(zip(gts_u8, rows4)):
        if not (0 <= r0 <= r1 <= H):
            raise ValueError(f"view {k}: window rows [{r0},{r1}) outside [0,{H})")
        if r1 == r0:
            keep.append(None)
            continue
        if not (r0 <= c0 <= c1 <= r1):
            raise ValueError(f"view {k}: counted rows [{c0},{c1}) must lie inside [{r0},{r1})")
        if not isinstance(gt, torch.Tensor) or gt.dtype != torch.uint8 or not gt.is_cuda:
            raise TypeError("gt windows must be CUDA uint8 tensors (3, rows, W)")
        if tuple(gt.shape) != (3, r1 - r0, W):
            raise ValueError(f"gt window {k} must be (3,{r1 - r0},{W}), got {tuple(gt.shape)}")
        keep.append(gt.contiguous())
    flat = _i32_array([v for r in rows4 for v in r])
    gptr = (C.c_void_p * B)(*[None if g is None else g.data_ptr() for g in keep])
    out = torch.empty((B, 3, 3), dtype=torch.float64, device=images.device)
    _lib.call("gs_metrics_batched", B, H, W, flat, images.data_ptr(), gptr, 1 if saved else 0, out.data_ptr(), _stream())
    return out


def get_local2j_ids_bool(image_height, image_width, rank, world_size, means2D, radii, dist_global_strategy,
                         cuda_args=None):
    """(P, world_size) bool: does splat i touch rank j's flattened tile range.  `rank` is unused (kept for
    signature parity with workload_division.py:727-738)."""
    means2D = _f32c(means2D.detach(), "means2D")
    radii = radii.to(torch.int32).contiguous()
    strat = dist_global_strategy.to(device=means2D.device, dtype=torch.int32).contiguous()
    if strat.numel() != world_size + 1:
        raise ValueError("dist_global_strategy must have world_size+1 entries")
    P = means2D.shape[0]
    out = torch.empty((P, world_size), dtype=torch.bool, device=means2D.device)
    _lib.call("gs_get_local2j_ids_bool", P, int(image_height), int(image_width), int(world_size), means2D.data_ptr(),
              radii.data_ptr(), strat.data_ptr(), out.data_ptr(), _stream())
    return out


def get_local2j_ids_bool_adjust_mode6(image_height, image_width, rank, world_size, means2D, radii, rectangles,
                                      cuda_args=None):
    """Legacy variant (workload_division.py:471-484): rank j owns tile rectangle (y_l, y_r, x_l, x_r)."""
    means2D = _f32c(means2D.detach(), "means2D")
    radii = radii.to(torch.int32).contiguous()
    rects = rectangles.to(device=means2D.device, dtype=torch.int32).contiguous()
    P = means2D.shape[0]
    out = torch.empty((P, world_size), dtype=torch.bool, device=means2D.device)
    _lib.call("gs_get_local2j_ids_bool_rects", P, int(image_height), int(image_width), int(world_size),
              means2D.data_ptr(), radii.data_ptr(), rects.data_ptr(), out.data_ptr(), _stream())
    return out


def get_block_XY():
    """(BLOCK_X, BLOCK_Y, ONE_DIM_BLOCK_SIZE) as compiled into the library (arguments/__init__.py:254-257)."""
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    _lib.call("gs_get_block_xy", C.byref(a), C.byref(b), C.byref(c))
    return a.value, b.value, c.value


class _FusedL1SSIM(torch.autograd.Function):
    """Per-strip (Ll1, ssim) of loss_distribution.py:2536-2585 in two kernels instead of ~20."""

    @staticmethod
    def forward(ctx, image, gt_u8, row0, row1, crow0, crow1):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        image = _f32c(image, "image")
        if gt_u8.dtype != torch.uint8 or not gt_u8.is_cuda:
            raise TypeError("gt strip must be a CUDA uint8 tensor (3, rows, W)")
        gt_u8 = gt_u8.contiguous()
        _, H, W = image.shape
        rows = row1 - row0
        if tuple(gt_u8.shape) != (3, rows, W):
            raise ValueError(f"gt strip must be (3,{rows},{W}), got {tuple(gt_u8.shape)}")
        tb = _lib.query("gs_loss_temp_bytes", rows, W)
        temp = torch.empty((tb,), dtype=torch.uint8, device=image.device)
        out = torch.empty((2,), dtype=torch.float32, device=image.device)
        _lib.call("gs_loss_forward", H, W, row0, row1, crow0, crow1, image.data_ptr(), gt_u8.data_ptr(), out.data_ptr(),
                  temp.data_ptr(), tb, _stream())
        ctx.rows = (row0, row1, crow0, crow1)
        ctx.save_for_backward(image, gt_u8, temp)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, g_l1, g_ssim):
        image, gt_u8, temp = ctx.saved_tensors
        _, H, W = image.shape
        row0, row1, crow0, crow1 = ctx.rows
        dev = image.device
        g_l1 = torch.zeros((), device=dev) if g_l1 is None else g_l1
        g_ssim = torch.zeros((), device=dev) if g_ssim is None else g_ssim
        g_l1, g_ssim = g_l1.to(torch.float32).contiguous(), g_ssim.to(torch.float32).contiguous()
        d_image = torch.empty_like(image)
        _lib.call("gs_loss_backward", H, W, row0, row1, crow0, crow1, image.data_ptr(), gt_u8.data_ptr(),
                  temp.data_ptr(), g_l1.data_ptr(), g_ssim.data_ptr(), d_image.data_ptr(), _stream())
        return d_image, None, None, None, None, None


def fused_l1_ssim(image, gt_u8, row0, row1, count_row0=None, count_row1=None):
    """-> (Ll1, ssim_loss) 0-dim tensors, both normalised by 3*H*W of the FULL image.
    Rows [row0,row1) of `image` (and the (3,row1-row0,W) uint8 `gt_u8`) form the window the 11x11 SSIM filter sees;
    only rows [count_row0,count_row1) (default: the whole window) are summed -- pass a window widened by exchanged halo
    rows to make strip losses add up to the full-image loss (border-pixel exchange, loss_distribution.py:601-972)."""
    c0 = int(row0) if count_row0 is None else int(count_row0)
    c1 = int(row1) if count_row1 is None else int(count_row1)
    return _FusedL1SSIM.apply(image, gt_u8, int(row0), int(row1), c0, c1)


_LOSS_W = {}


class _FusedLoss(torch.autograd.Function):
    """(1 - lambda) Ll1 + lambda (1 - ssim) of one strip as ONE autograd node (train_internal.py:166-189 forms it with five
    elementwise kernels and as many in the backward): the two sums come out of gs_loss_forward, the combination is one dot
    product with a cached weight vector, and the backward hands (g (1 - lambda), -g lambda) to gs_loss_backward."""

    @staticmethod
    def forward(ctx, image, gt_u8, row0, row1, crow0, crow1, lambda_dssim):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        image = _f32c(image, "image")
        if gt_u8.dtype != torch.uint8 or not gt_u8.is_cuda:
            raise TypeError("gt strip must be a CUDA uint8 tensor (3, rows, W)")
        gt_u8 = gt_u8.contiguous()
        _, H, W = image.shape
        rows = row1 - row0
        if tuple(gt_u8.shape) != (3, rows, W):
            raise ValueError(f"gt strip must be (3,{rows},{W}), got {tuple(gt_u8.shape)}")
        key = (image.device, float(lambda_dssim))
        if key not in _LOSS_W:
            _LOSS_W[key] = torch.tensor([1.0 - lambda_dssim, -lambda_dssim], dtype=torch.float32, device=image.device)
        w = _LOSS_W[key]
        tb = _lib.query("gs_loss_temp_bytes", rows, W)
        temp = torch.empty((tb,), dtype=torch.uint8, device=image.device)
        out = torch.empty((2,), dtype=torch.float32, device=image.device)
        _lib.call("gs_loss_forward", H, W, row0, row1, crow0, crow1, image.data_ptr(), gt_u8.data_ptr(), out.data_ptr(),
                  temp.data_ptr(), tb, _stream())
        ctx.rows, ctx.w = (row0, row1, crow0, crow1), w
        ctx.save_for_backward(image, gt_u8, temp)
        return torch.dot(out, w) + float(lambda_dssim)

    @staticmethod
    def backward(ctx, g):
        image, gt_u8, temp = ctx.saved_tensors
        _, H, W = image.shape
        row0, row1, crow0, crow1 = ctx.rows
        if g is None:
            return None, None, None, None, None, None, None
        gw = (g.to(torch.float32) * ctx.w).contiguous()      # (g (1 - lambda), -g lambda)
        d_image = torch.empty_like(image)
        _lib.call("gs_loss_backward", H, W, row0, row1, crow0, crow1, image.data_ptr(), gt_u8.data_ptr(),
                  temp.data_ptr(), gw.data_ptr(), gw.data_ptr() + 4, d_image.data_ptr(), _stream())
        return d_image, None, None, None, None, None, None


def fused_loss(image, gt_u8, row0, row1, lambda_dssim, count_row0=None, count_row1=None):
    """-> 0-dim loss (1 - lambda) Ll1 + lambda (1 - ssim) of the strip rows [row0, row1) (same window / count-row
    semantics as fused_l1_ssim)."""
    c0 = int(row0) if count_row0 is None else int(count_row0)
    c1 = int(row1) if count_row1 is None else int(count_row1)
    return _FusedLoss.apply(image, gt_u8, int(row0), int(row1), c0, c1, float(lambda_dssim))


# ---------------------------------------------------------------------------------------------------------
# legacy tile-mask / tile-exchange helpers (SURVEY.md 8a rows L3-L4; never called by the shipped trainer)
# ---------------------------------------------------------------------------------------------------------
def _mask_u8(m):
    if not m.is_cuda:
        raise ValueError("compute_locally must be a CUDA tensor")
    m = m.contiguous()
    return m.view(torch.uint8) if m.dtype == torch.bool else m.to(torch.uint8)


def get_touched_locally(compute_locally, image_height, image_width, extension_distance):
    """(TILE_Y, TILE_X) bool: tiles within `extension_distance` tiles of a locally computed tile
    (/root/reference/gaussian_renderer/loss_distribution.py:136-141)."""
    cl = _mask_u8(compute_locally)
    ty, tx = (int(image_height) + BLOCK_Y - 1) // BLOCK_Y, (int(image_width) + BLOCK_X - 1) // BLOCK_X
    if cl.numel() != ty * tx:
        raise ValueError("compute_locally does not match the image's tile grid")
    out = torch.empty((ty, tx), dtype=torch.bool, device=cl.device)
    _lib.call("gs_get_touched_locally", ty, tx, int(extension_distance), cl.data_ptr(), out.data_ptr(), _stream())
    return out


def get_pixels_compute_locally_and_in_rect(compute_locally, image_height, image_width, min_y, max_y, min_x, max_x):
    """(max_y-min_y, max_x-min_x) bool pixel mask: is the pixel's tile computed locally (loss_distribution.py:205-213)."""
    cl = _mask_u8(compute_locally)
    out = torch.empty((int(max_y) - int(min_y), int(max_x) - int(min_x)), dtype=torch.bool, device=cl.device)
    _lib.call("gs_get_pixels_compute_locally_and_in_rect", int(image_height), int(image_width), cl.data_ptr(), int(min_y),
              int(max_y), int(min_x), int(max_x), out.data_ptr(), _stream())
    return out


class _LoadImageTilesByPos(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rect, pos, H, W, pixels_rect, tiles_rect):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        rect = _f32c(rect, "local_image_rect")
        pos = pos.to(device=rect.device, dtype=torch.int64).contiguous().reshape(-1, 2)
        n = pos.shape[0]
        _, rh, rw = rect.shape
        tiles = torch.empty((n, 3, BLOCK_Y, BLOCK_X), dtype=torch.float32, device=rect.device)
        _lib.call("gs_image_tiles_gather", n, pos.data_ptr(), rect.data_ptr(), rh, rw, int(pixels_rect[0]),
                  int(pixels_rect[2]), int(H), int(W), tiles.data_ptr(), _stream())
        ctx.save_for_backward(pos)
        ctx.meta = (rh, rw, int(pixels_rect[0]), int(pixels_rect[2]), int(H), int(W))
        return tiles

    @staticmethod
    def backward(ctx, g):
        (pos,) = ctx.saved_tensors
        rh, rw, y0, x0, H, W = ctx.meta
        if g is None:
            return None, None, None, None, None, None
        g = _f32c(g, "grad")
        out = torch.zeros((3, rh, rw), dtype=torch.float32, device=g.device)
        _lib.call("gs_image_tiles_scatter_add", pos.shape[0], pos.data_ptr(), g.data_ptr(), rh, rw, y0, x0, H, W,
                  out.data_ptr(), _stream())
        return out, None, None, None, None, None


class _MergeImageTilesByPos(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, tiles, H, W, pixels_rect, tiles_rect):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        tiles = _f32c(tiles, "tiles")
        pos = pos.to(device=tiles.device, dtype=torch.int64).contiguous().reshape(-1, 2)
        rh, rw = int(pixels_rect[1]) - int(pixels_rect[0]), int(pixels_rect[3]) - int(pixels_rect[2])
        out = torch.zeros((3, rh, rw), dtype=torch.float32, device=tiles.device)
        _lib.call("gs_image_tiles_scatter_add", pos.shape[0], pos.data_ptr(), tiles.data_ptr(), rh, rw,
                  int(pixels_rect[0]), int(pixels_rect[2]), int(H), int(W), out.data_ptr(), _stream())
        ctx.save_for_backward(pos)
        ctx.meta = (rh, rw, int(pixels_rect[0]), int(pixels_rect[2]), int(H), int(W))
        return out

    @staticmethod
    def backward(ctx, g):
        (pos,) = ctx.saved_tensors
        rh, rw, y0, x0, H, W = ctx.meta
        if g is None:
            return None, None, None, None, None, None
        g = _f32c(g, "grad")
        n = pos.shape[0]
        tiles = torch.empty((n, 3, BLOCK_Y, BLOCK_X), dtype=torch.float32, device=g.device)
        _lib.call("gs_image_tiles_gather", n, pos.data_ptr(), g.data_ptr(), rh, rw, y0, x0, H, W, tiles.data_ptr(),
                  _stream())
        return None, tiles, None, None, None, None


def load_image_tiles_by_pos(local_image_rect, all_pos_send_to_j, image_height, image_width, touched_pixels_rect,
                            touched_tiles_rect):
    """(3,h,w) local rect -> (n,3,16,16) tiles at GLOBAL tile positions (n,2); differentiable
    (/root/reference/gaussian_renderer/loss_distribution.py:168-175)."""
    return _LoadImageTilesByPos.apply(local_image_rect, all_pos_send_to_j, image_height, image_width,
                                      touched_pixels_rect, touched_tiles_rect)


def merge_image_tiles_by_pos(all_pos_recv_from_i, all_tiles_recv_from_i, image_height, image_width, touched_pixels_rect,
                             touched_tiles_rect):
    """(n,3,16,16) tiles at GLOBAL tile positions -> (3,h,w) local rect, zero elsewhere; differentiable
    (loss_distribution.py:188-195)."""
    return _MergeImageTilesByPos.apply(all_pos_recv_from_i, all_tiles_recv_from_i, image_height, image_width,
                                       touched_pixels_rect, touched_tiles_rect)


# ---------------------------------------------------------------------------------------------------------
# batched preprocess: all B cameras of a step in one launch
# ---------------------------------------------------------------------------------------------------------
def pack_cameras(settings_list):
    """(B,40) float32 device tensor: viewmatrix[16], projmatrix[16], campos[3], tanfovx, tanfovy, 3 pad per camera."""
    rows = []
    for rs in settings_list:
        dev = rs.viewmatrix.device
        tail = torch.tensor([float(rs.tanfovx), float(rs.tanfovy), 0.0, 0.0, 0.0], dtype=torch.float32, device=dev)
        rows.append(torch.cat([rs.viewmatrix.reshape(-1).float(), rs.projmatrix.reshape(-1).float(),
                               rs.campos.reshape(-1).float(), tail]))
    return torch.stack(rows).contiguous()


class _PreprocessBatched(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, f_dc, f_rest, scaling, rotation, opacity, cams, meta):
        ctx.set_materialize_grads(False)   # undefined output gradients arrive as None, not as zero-filled tensors
        xyz, f_dc, f_rest = _f32c(xyz, "_xyz"), _f32c(f_dc, "_features_dc"), _f32c(f_rest, "_features_rest")
        scaling, rotation, opacity = _f32c(scaling, "_scaling"), _f32c(rotation, "_rotation"), _f32c(opacity, "_opacity")
        cams = _f32c(cams, "cams")
        P, B = xyz.shape[0], cams.shape[0]
        if tuple(f_dc.shape) != (P, 1, 3) or tuple(f_rest.shape) != (P, 15, 3) or cams.shape[1] != 40:
            raise ValueError("features must be (P,1,3)/(P,15,3) and cams (B,40)")
        W, H, D, mod = meta
        dev = xyz.device
        means2D = torch.empty((B, P, 2), dtype=torch.float32, device=dev)
        depths = torch.empty((B, P), dtype=torch.float32, device=dev)
        radii = torch.empty((B, P), dtype=torch.int32, device=dev)
        conic_opacity = torch.empty((B, P, 4), dtype=torch.float32, device=dev)
        rgb = torch.empty((B, P, 3), dtype=torch.float32, device=dev)
        clamped = torch.empty((B, P), dtype=torch.uint8, device=dev)
        _lib.call("gs_preprocess_forward_batched", B, P, int(D), xyz.data_ptr(), f_dc.data_ptr(), f_rest.data_ptr(),
                  scaling.data_ptr(), float(mod), rotation.data_ptr(), opacity.data_ptr(), cams.data_ptr(), int(W),
                  int(H), means2D.data_ptr(), depths.data_ptr(), radii.data_ptr(), conic_opacity.data_ptr(),
                  rgb.data_ptr(), clamped.data_ptr(), _stream())
        ctx.meta = meta
        ctx.save_for_backward(xyz, f_dc, f_rest, scaling, rotation, opacity, cams, radii, clamped)
        ctx.mark_non_differentiable(radii, depths)
        return means2D, rgb, conic_opacity, radii, depths

    @staticmethod
    def backward(ctx, g_means2D, g_rgb, g_conic_opacity, _g_radii, _g_depths):
        xyz, f_dc, f_rest, scaling, rotation, opacity, cams, radii, clamped = ctx.saved_tensors
        W, H, D, mod = ctx.meta
        P, B = xyz.shape[0], cams.shape[0]
        dev = xyz.device

        def z(g, shape):
            return torch.zeros(shape, dtype=torch.float32, device=dev) if g is None else _f32c(g, "grad")

        g_means2D, g_rgb, g_conic_opacity = z(g_means2D, (B, P, 2)), z(g_rgb, (B, P, 3)), z(g_conic_opacity, (B, P, 4))
        d = [torch.empty_like(t) for t in (xyz, f_dc, f_rest, scaling, rotation, opacity)]
        _lib.call("gs_preprocess_backward_batched", B, P, int(D), xyz.data_ptr(), f_dc.data_ptr(), f_rest.data_ptr(),
                  scaling.data_ptr(), float(mod), rotation.data_ptr(), opacity.data_ptr(), cams.data_ptr(), int(W),
                  int(H), radii.data_ptr(), clamped.data_ptr(), g_means2D.data_ptr(), g_conic_opacity.data_ptr(),
                  g_rgb.data_ptr(), d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), d[4].data_ptr(),
                  d[5].data_ptr(), _stream())
        return d[0], d[1], d[2], d[3], d[4], d[5], None, None


def preprocess_gaussians_batched(xyz, features_dc, features_rest, scaling, rotation, opacity, cams, image_width,
                                 image_height, sh_degree, scale_modifier=1.0):
    """All B cameras at once from the RAW GaussianModel parameters.  cams: pack_cameras(...) (B,40).
    -> (means2D (B,P,2), rgb (B,P,3), conic_opacity (B,P,4), radii (B,P) int32, depths (B,P)); slice k equals the
    single-camera operator's output for camera k."""
    return _PreprocessBatched.apply(xyz, features_dc, features_rest, scaling, rotation, opacity, cams,
                                    (int(image_width), int(image_height), int(sh_degree), float(scale_modifier)))
