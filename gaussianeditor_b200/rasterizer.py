"""Drop-in replacement of the reference's ``diff_gaussian_rasterization`` Python package.

Same public names, argument meaning, return values and error messages as
/root/reference/gaussiansplatting/submodules/diff-gaussian-rasterization/diff_gaussian_rasterization/__init__.py
(``GaussianRasterizationSettings`` :228-240, ``GaussianRasterizer`` :243-364, ``rasterize_gaussians`` :26-47,
``_RasterizeGaussians`` :50-225), backed by the sm_100a C-ABI library instead of the ``_C`` pybind module.

Differences a caller can observe (all documented in DESIGN.md):
  * kernels run on PyTorch's CURRENT stream (the reference always used the legacy default stream);
  * the only host synchronisation per forward is one stream sync to read ``num_rendered``;
  * gradient tensors are written completely by the kernels (no separate zero-fill passes);
  * ``debug=True`` synchronises after every launch and raises on the first CUDA error, but does not write the
    reference's ``snapshot_*.dump`` files.
"""
from __future__ import annotations

import ctypes as C
import threading
import time
from typing import NamedTuple

import torch
import torch.nn as nn

from . import _lib


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


_size_cache: dict = {}
_pinned: dict = {}
_r_hint: dict = {}          # (device, P, W, H) -> largest num_rendered seen recently
SPECULATIVE = True          # launch the second forward half before num_rendered is known (see _forward_impl)
SPEC_STATS = {"launched": 0, "missed": 0}   # speculative second halves launched / redone because the guess was too small


def _f32c(t: torch.Tensor, device) -> torch.Tensor:
    """float32, contiguous, on `device`, 16-byte aligned storage."""
    if t.dtype != torch.float32 or t.device != device or not t.is_contiguous():
        t = t.to(device=device, dtype=torch.float32).contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t


def _ptr(t):
    return None if t is None or t.numel() == 0 else C.c_void_p(t.data_ptr())


def _bounded_put(d: dict, key, value, limit: int = 64):
    """Densification changes P every few hundred steps: keep the per-(P, W, H) dictionaries from growing forever."""
    if key not in d and len(d) >= limit:
        d.pop(next(iter(d)))
    d[key] = value


def _geometry_bytes(lib, P):
    key = ("g", P)
    if key not in _size_cache:
        n = lib.gsr_geometry_bytes(P)
        if n == 0:
            _lib.check(-2, "gsr_geometry_bytes")
        _bounded_put(_size_cache, key, n)
    return _size_cache[key]


def _pinned_i32(device):
    """One pinned count word per (device, stream, host thread): two threads driving forwards on the same stream (e.g. the
    autograd engine thread re-running a checkpointed forward) must not poll each other's word."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, threading.get_ident())
    if key not in _pinned:
        _bounded_put(_pinned, key, torch.zeros(1, dtype=torch.int32).pin_memory(), limit=256)
    return _pinned[key]


def _wait_count(pinned: torch.Tensor, waiter) -> int:
    """num_rendered arrives in a pinned host word (preset to -1) through an async copy that the library issues right
    behind the preprocess kernel, i.e. BEFORE the depth sort it has already queued: spinning on the word hands the
    count to the host while the GPU is still busy, instead of sleeping until the whole first half has drained.
    Falls back to `waiter()` (event / stream synchronize) after 2 ms."""
    t0 = time.perf_counter()
    while int(pinned[0]) < 0:
        if time.perf_counter() - t0 > 2e-3:
            waiter()
            break
    return int(pinned[0])


def _make_settings(rs: GaussianRasterizationSettings, M: int, device, keep: list) -> _lib.Settings:
    bg = _f32c(rs.bg, device); view = _f32c(rs.viewmatrix, device)
    proj = _f32c(rs.projmatrix, device); campos = _f32c(rs.campos, device)
    keep += [bg, view, proj, campos]
    return _lib.Settings(int(rs.image_height), int(rs.image_width), float(rs.tanfovx), float(rs.tanfovy),
                         float(rs.scale_modifier), int(rs.sh_degree), int(M), int(bool(rs.prefiltered)),
                         int(bool(rs.debug)), bg.data_ptr(), view.data_ptr(), proj.data_ptr(), campos.data_ptr())


def _make_cloud(P, means3D, opacities, sh, colors_precomp, scales, rotations, cov3Ds_precomp) -> _lib.Cloud:
    return _lib.Cloud(P, _ptr(means3D), _ptr(opacities), _ptr(sh), _ptr(colors_precomp), _ptr(scales),
                      _ptr(rotations), _ptr(cov3Ds_precomp))


class _ForwardState:
    """What the forward leaves behind for backward / apply_weights / parity tests."""
    __slots__ = ("geom", "binning", "img", "radii", "num_rendered", "cap", "P", "M", "W", "H")


def _forward_impl(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, rs, *, render=True,
                  raw_rest=None):
    """Both forward halves. With ``raw_rest`` (features_rest [P,K,3]) the call is the fused-activation variant:
    ``sh`` is features_dc [P,1,3] and opacities / scales / rotations are the raw parameters."""
    lib = _lib.load()
    if means3D.dim() != 2 or means3D.size(1) != 3:
        raise RuntimeError("means3D must have dimensions (num_points, 3)")  # rasterize_points.cu:46-48
    if not means3D.is_cuda:
        raise RuntimeError("the B200 rasterizer needs CUDA tensors (there is no CPU path)")
    device = means3D.device
    P = means3D.size(0)
    H, W = int(rs.image_height), int(rs.image_width)
    M = sh.size(1) if sh.numel() != 0 else 0
    raw = raw_rest is not None
    if raw:
        M = 1 + raw_rest.size(1)
    with torch.cuda.device(device):
        if raw:
            raw_rest = _f32c(raw_rest, device)
        means3D = _f32c(means3D, device); opacities = _f32c(opacities, device)
        sh = _f32c(sh, device); colors_precomp = _f32c(colors_precomp, device)
        scales = _f32c(scales, device); rotations = _f32c(rotations, device)
        cov3Ds_precomp = _f32c(cov3Ds_precomp, device)
        keep = []
        s = _make_settings(rs, M, device, keep)
        c = _make_cloud(P, means3D, opacities, sh, colors_precomp, scales, rotations, cov3Ds_precomp)
        stream = torch.cuda.current_stream(device)
        st = C.c_void_p(stream.cuda_stream)
        u8 = dict(dtype=torch.uint8, device=device)
        state = _ForwardState()
        state.P, state.M, state.W, state.H = P, M, W, H
        state.radii = torch.empty(P, dtype=torch.int32, device=device)
        gbytes = _geometry_bytes(lib, P) if P > 0 else 0
        state.geom = torch.empty(gbytes, **u8)
        pinned = _pinned_i32(device)
        pinned[0] = -1
        if raw:
            rc = _lib.RawCloud(P, _ptr(means3D), _ptr(opacities), _ptr(sh), _ptr(raw_rest), _ptr(scales), _ptr(rotations))
            _lib.check(lib.gsr_forward_preprocess_raw(C.byref(s), C.byref(rc), _ptr(state.geom), gbytes,
                                                      _ptr(state.radii), C.c_void_p(pinned.data_ptr()), st),
                       "gsr_forward_preprocess_raw")
        else:
            _lib.check(lib.gsr_forward_preprocess(C.byref(s), C.byref(c), _ptr(state.geom), gbytes, _ptr(state.radii),
                                                  C.c_void_p(pinned.data_ptr()), st), "gsr_forward_preprocess")
        ibytes = lib.gsr_image_bytes(W, H)
        state.img = torch.empty(ibytes, **u8)
        color = depth = None
        if render:
            color = torch.empty(3, H, W, dtype=torch.float32, device=device)
            depth = torch.empty(1, H, W, dtype=torch.float32, device=device)
        key = (device.index, P, W, H)
        hint = _r_hint.get(key)
        done = False
        if SPECULATIVE and render and P > 0 and hint:
            # The count of (Gaussian, tile) instances is only known on the device at this point. Instead of idling
            # the GPU while the host fetches it (the reference blocks in cudaMemcpy), enqueue the second half now for
            # a guessed capacity, THEN wait for the count: the GPU keeps working while the host waits. A wrong guess
            # (count > capacity) is detected below and the second half is redone with the exact size.
            ev = torch.cuda.Event()
            ev.record(stream)
            cap = int(hint * 1.25) + 4096
            bbytes = lib.gsr_binning_bytes(P, cap, W, H)
            state.binning = torch.empty(bbytes, **u8)
            _lib.check(lib.gsr_forward_render_speculative(C.byref(s), C.byref(c), cap, _ptr(state.geom), gbytes,
                                                          _ptr(state.binning), bbytes, _ptr(state.img), ibytes,
                                                          _ptr(state.radii), _ptr(color), _ptr(depth), st),
                       "gsr_forward_render_speculative")
            R = _wait_count(pinned, ev.synchronize)
            SPEC_STATS["launched"] += 1
            if R <= cap:
                state.num_rendered, state.cap, done = R, cap, True
            else:
                SPEC_STATS["missed"] += 1
        if not done:
            R = _wait_count(pinned, stream.synchronize)
            state.num_rendered = state.cap = R
            bbytes = lib.gsr_binning_bytes(P, R, W, H) if R > 0 else 0
            state.binning = torch.empty(bbytes, **u8)
            if render:
                _lib.check(lib.gsr_forward_render(C.byref(s), C.byref(c), R, _ptr(state.geom), gbytes,
                                                  _ptr(state.binning), bbytes, _ptr(state.img), ibytes,
                                                  _ptr(state.radii), _ptr(color), _ptr(depth), st), "gsr_forward_render")
        if P > 0:
            _bounded_put(_r_hint, key, max(R, int(0.9 * _r_hint.get(key, 0))))
    inputs = (means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp)
    if raw:
        inputs = inputs + (raw_rest,)
    return color, depth, state, inputs


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings, return_alpha=False, camera_grad=False, depth_grad=False):
    if camera_grad:   # the camera arrays become autograd inputs of the node (they are read from the settings as usual)
        rs = raster_settings
        return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                         cov3Ds_precomp, rs, return_alpha, depth_grad, rs.viewmatrix, rs.projmatrix,
                                         rs.campos)
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                     cov3Ds_precomp, raster_settings, return_alpha, depth_grad)


def _alpha_image(lib, state, device):
    """alpha = 1 - final_T as a [1,H,W] tensor (gsr_alpha_image; final_T is the reference's accum_alpha)."""
    alpha = torch.zeros(1, state.H, state.W, dtype=torch.float32, device=device)
    if state.P > 0 and state.W * state.H > 0:
        st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        _lib.check(lib.gsr_alpha_image(_ptr(state.img), state.img.numel(), state.W, state.H, _ptr(alpha), st),
                   "gsr_alpha_image")
    return alpha


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                raster_settings, return_alpha=False, depth_grad=False, viewmatrix=None, projmatrix=None, campos=None):
        color, depth, state, inputs = _forward_impl(means3D, sh, colors_precomp, opacities, scales, rotations,
                                                    cov3Ds_precomp, raster_settings)
        ctx.raster_settings = raster_settings
        ctx.camera_grad = viewmatrix is not None
        ctx.depth_grad = bool(depth_grad)
        ctx.n_inputs = 11 + (3 if ctx.camera_grad else 0)
        ctx.state = state
        ctx.save_for_backward(*inputs, state.radii, state.geom, state.binning, state.img)
        ctx.mark_non_differentiable(state.radii)
        _RasterizeGaussians.last_state = state  # for parity tests / instrumentation only
        if return_alpha:   # opt-in fourth output (not in the reference's tuple): alpha = 1 - final_T, differentiable
            with torch.cuda.device(means3D.device):
                return color, state.radii, depth, _alpha_image(_lib.load(), state, means3D.device)
        return color, state.radii, depth

    @staticmethod
    def backward(ctx, grad_out_color, grad_radii, grad_depth, grad_alpha=None):
        lib = _lib.load()
        rs = ctx.raster_settings
        state = ctx.state
        (means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, radii, geom, binning,
         img) = ctx.saved_tensors
        device = means3D.device
        P, M, W, H = state.P, state.M, state.W, state.H
        with torch.cuda.device(device):
            grad_out_color = _f32c(grad_out_color, device)
            f32 = dict(dtype=torch.float32, device=device)
            dL_dmeans3D = torch.empty(P, 3, **f32); dL_dmeans2D = torch.empty(P, 3, **f32)
            dL_dcolors = torch.empty(P, 3, **f32); dL_dopacity = torch.empty(P, 1, **f32)
            dL_dcov3D = torch.empty(P, 6, **f32); dL_dsh = torch.empty(P, M, 3, **f32)
            dL_dscales = torch.empty(P, 3, **f32); dL_drotations = torch.empty(P, 4, **f32)
            if P > 0:
                keep = []
                s = _make_settings(rs, M, device, keep)
                c = _make_cloud(P, means3D, opacities, sh, colors_precomp, scales, rotations, cov3Ds_precomp)
                sbytes = lib.gsr_backward_scratch_bytes(P)
                scratch = torch.empty(sbytes, dtype=torch.uint8, device=device)
                gr = _lib.Grads(_ptr(dL_dmeans3D), _ptr(dL_dmeans2D), _ptr(dL_dcolors), _ptr(dL_dopacity),
                                _ptr(dL_dcov3D), _ptr(dL_dsh), _ptr(dL_dscales), _ptr(dL_drotations))
                st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
                cam = None
                if ctx.camera_grad:
                    d_view = torch.empty(16, **f32); d_proj = torch.empty(16, **f32); d_cam = torch.empty(3, **f32)
                    cbytes = lib.gsr_camera_scratch_bytes(P)
                    cscratch = torch.empty(cbytes, dtype=torch.uint8, device=device)
                    cam = _lib.CameraGrads(_ptr(d_view), _ptr(d_proj), _ptr(d_cam), _ptr(cscratch), cbytes)
                    cam_grads = (d_view.view(rs.viewmatrix.shape), d_proj.view(rs.projmatrix.shape),
                                 d_cam.view(rs.campos.shape))
                if ctx.depth_grad:   # one entry point for every combination with the alpha and camera gradients
                    ga = None if grad_alpha is None else _f32c(grad_alpha, device)
                    gd = _f32c(grad_depth, device)
                    _lib.check(lib.gsr_backward_depth(C.byref(s), C.byref(c), state.cap, _ptr(geom), geom.numel(),
                                                      _ptr(binning), binning.numel(), _ptr(img), img.numel(),
                                                      _ptr(radii), _ptr(grad_out_color), _ptr(ga), _ptr(gd),
                                                      _ptr(scratch), sbytes, C.byref(gr),
                                                      None if cam is None else C.byref(cam), st), "gsr_backward_depth")
                elif ctx.camera_grad:
                    ga = None if grad_alpha is None else _f32c(grad_alpha, device)
                    _lib.check(lib.gsr_backward_camera(C.byref(s), C.byref(c), state.cap, _ptr(geom), geom.numel(),
                                                       _ptr(binning), binning.numel(), _ptr(img), img.numel(),
                                                       _ptr(radii), _ptr(grad_out_color), _ptr(ga), _ptr(scratch), sbytes,
                                                       C.byref(gr), C.byref(cam), st), "gsr_backward_camera")
                elif grad_alpha is not None:
                    grad_alpha = _f32c(grad_alpha, device)
                    _lib.check(lib.gsr_backward_alpha(C.byref(s), C.byref(c), state.cap, _ptr(geom), geom.numel(),
                                                      _ptr(binning), binning.numel(), _ptr(img), img.numel(),
                                                      _ptr(radii), _ptr(grad_out_color), _ptr(grad_alpha),
                                                      _ptr(scratch), sbytes, C.byref(gr), st), "gsr_backward_alpha")
                else:
                    _lib.check(lib.gsr_backward(C.byref(s), C.byref(c), state.cap, _ptr(geom), geom.numel(),
                                                _ptr(binning), binning.numel(), _ptr(img), img.numel(), _ptr(radii),
                                                _ptr(grad_out_color), _ptr(scratch), sbytes, C.byref(gr), st),
                               "gsr_backward")
                if scales.numel() == 0:  # cov3D_precomp path: the reference leaves these at their zero-fill
                    dL_dscales.zero_(); dL_drotations.zero_()
        # same slots as the reference (__init__.py:213-223); autograd drops grads of inputs that do not need one
        grads = (dL_dmeans3D, dL_dmeans2D, dL_dsh, dL_dcolors, dL_dopacity, dL_dscales, dL_drotations, dL_dcov3D,
                 None, None, None)
        if ctx.camera_grad:
            if P == 0:
                z = lambda t: torch.zeros_like(t, dtype=torch.float32)
                cam_grads = (z(rs.viewmatrix), z(rs.projmatrix), z(rs.campos))
            grads = grads + cam_grads
        return grads


class _RasterizeGaussiansRaw(torch.autograd.Function):
    """Fused-activation variant (SURVEY 8(f-3), gsr_forward_preprocess_raw / gsr_backward_raw): takes the scene model's
    raw parameters, gradients come back w.r.t. them."""

    @staticmethod
    def forward(ctx, means3D, means2D, opacity_logits, features_dc, features_rest, log_scales, raw_rotations,
                raster_settings, depth_grad=False):
        empty = torch.empty(0, dtype=torch.float32, device=means3D.device)
        color, depth, state, inputs = _forward_impl(means3D, features_dc, empty, opacity_logits, log_scales,
                                                    raw_rotations, empty, raster_settings, raw_rest=features_rest)
        ctx.raster_settings = raster_settings
        ctx.depth_grad = bool(depth_grad)
        ctx.state = state
        (m3, dc, _, op, sc, ro, _, rest) = inputs
        ctx.save_for_backward(m3, dc, rest, op, sc, ro, state.radii, state.geom, state.binning, state.img)
        ctx.mark_non_differentiable(state.radii)
        _RasterizeGaussians.last_state = state
        return color, state.radii, depth

    @staticmethod
    def backward(ctx, grad_out_color, grad_radii, grad_depth):
        lib = _lib.load()
        rs, state = ctx.raster_settings, ctx.state
        (means3D, dc, rest, logits, log_scales, raw_rot, radii, geom, binning, img) = ctx.saved_tensors
        device = means3D.device
        P, M = state.P, state.M
        with torch.cuda.device(device):
            grad_out_color = _f32c(grad_out_color, device)
            f32 = dict(dtype=torch.float32, device=device)
            d_m3 = torch.empty(P, 3, **f32); d_m2 = torch.empty(P, 3, **f32); d_op = torch.empty(P, 1, **f32)
            d_dc = torch.empty(P, 1, 3, **f32); d_rest = torch.empty(P, M - 1, 3, **f32)
            d_sc = torch.empty(P, 3, **f32); d_ro = torch.empty(P, 4, **f32)
            if P > 0:
                keep = []
                s = _make_settings(rs, M, device, keep)
                rc = _lib.RawCloud(P, _ptr(means3D), _ptr(logits), _ptr(dc), _ptr(rest), _ptr(log_scales), _ptr(raw_rot))
                gr = _lib.RawGrads(_ptr(d_m3), _ptr(d_m2), _ptr(d_op), _ptr(d_dc), _ptr(d_rest), _ptr(d_sc), _ptr(d_ro))
                sbytes = lib.gsr_backward_scratch_bytes(P)
                scratch = torch.empty(sbytes, dtype=torch.uint8, device=device)
                st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
                if ctx.depth_grad:
                    gd = _f32c(grad_depth, device)
                    _lib.check(lib.gsr_backward_raw_depth(C.byref(s), C.byref(rc), state.cap, _ptr(geom), geom.numel(),
                                                          _ptr(binning), binning.numel(), _ptr(img), img.numel(),
                                                          _ptr(radii), _ptr(grad_out_color), _ptr(gd), _ptr(scratch),
                                                          sbytes, C.byref(gr), st), "gsr_backward_raw_depth")
                else:
                    _lib.check(lib.gsr_backward_raw(C.byref(s), C.byref(rc), state.cap, _ptr(geom), geom.numel(),
                                                    _ptr(binning), binning.numel(), _ptr(img), img.numel(), _ptr(radii),
                                                    _ptr(grad_out_color), _ptr(scratch), sbytes, C.byref(gr), st),
                               "gsr_backward_raw")
        return d_m3, d_m2, d_op, d_dc, d_rest, d_sc, d_ro, None, None


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings, return_alpha: bool = False, camera_grad: bool = False,
                 depth_grad: bool = False):
        """``return_alpha=True`` (opt-in, not in the reference) appends a fourth output to ``forward``: the alpha image
        ``1 - final_T`` [1,H,W] (the reference keeps final_T as ``accum_alpha`` but never returns it); it is
        differentiable like the colour.
        ``camera_grad=True`` (opt-in, not in the reference): ``raster_settings.viewmatrix / projmatrix / campos`` become
        differentiable inputs -- their ``.grad`` is filled by the backward (gsr_backward_camera), each array treated as an
        independent input exactly as the forward reads it.
        ``depth_grad=True`` (opt-in, not in the reference): the depth image (third output) becomes differentiable -- a
        loss on it reaches means3D, means2D, opacities, scales, rotations / cov3D_precomp (and the view matrix with
        ``camera_grad``) through gsr_backward_depth. Without the flag the gradient of the depth image is ignored, as in the
        reference: a loss on it trains nothing. Applies to ``forward`` and ``forward_raw``."""
        super().__init__()
        self.raster_settings = raster_settings
        self.return_alpha = bool(return_alpha)
        self.camera_grad = bool(camera_grad)
        self.depth_grad = bool(depth_grad)

    def forward_raw(self, means3D, means2D, opacity_logits, features_dc, features_rest, log_scales, raw_rotations):
        """Opt-in fused-activation call (not part of the reference API): the arguments are the scene model's raw
        parameters (``_xyz, _opacity, _features_dc, _features_rest, _scaling, _rotation``); sigmoid / exp / normalize
        and the SH concatenation happen inside the preprocess kernels. Same return tuple as ``forward``."""
        return _RasterizeGaussiansRaw.apply(means3D, means2D, opacity_logits, features_dc, features_rest, log_scales,
                                            raw_rotations, self.raster_settings, self.depth_grad)

    def markVisible(self, positions):
        # __init__.py:248-256 / rasterize_points.cu:159-175
        lib = _lib.load()
        with torch.no_grad():
            rs = self.raster_settings
            device = positions.device
            positions = _f32c(positions, device)
            P = positions.size(0)
            visible = torch.zeros(P, dtype=torch.bool, device=device)
            if P > 0:
                with torch.cuda.device(device):
                    view = _f32c(rs.viewmatrix, device); proj = _f32c(rs.projmatrix, device)
                    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
                    _lib.check(lib.gsr_mark_visible(P, _ptr(positions), _ptr(view), _ptr(proj), _ptr(visible), st),
                               "gsr_mark_visible")
        return visible

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        raster_settings = self.raster_settings

        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception("Please provide excatly one of either SHs or precomputed colors!")

        if ((scales is None or rotations is None) and cov3D_precomp is None) or (
            (scales is not None or rotations is not None) and cov3D_precomp is not None
        ):
            raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")

        empty = torch.empty(0, dtype=torch.float32, device=means3D.device)
        if shs is None:
            shs = empty
        if colors_precomp is None:
            colors_precomp = empty
        if scales is None:
            scales = empty
        if rotations is None:
            rotations = empty
        if cov3D_precomp is None:
            cov3D_precomp = empty

        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                   cov3D_precomp, raster_settings, self.return_alpha, self.camera_grad, self.depth_grad)

    def apply_weights(self, means3D, means2D, opacities, shs=None, weights=None, scales=None, rotations=None,
                      cov3Ds_precomp=None, cnt=None, image_weights=None):
        """Semantic tracing (__init__.py:311-364): in-place accumulation into ``weights`` [P,CH] float32 and
        ``cnt`` [P,1] int32 from the 2-D mask ``image_weights`` [CH,H,W]."""
        assert weights is not None
        assert cnt is not None
        assert image_weights is not None
        lib = _lib.load()
        rs = self.raster_settings
        device = means3D.device
        empty = torch.empty(0, dtype=torch.float32, device=device)
        if not (weights.is_cuda and weights.dtype == torch.float32 and weights.is_contiguous()):
            raise RuntimeError("weights must be a contiguous float32 CUDA tensor (it is updated in place)")
        if not (cnt.is_cuda and cnt.dtype == torch.int32 and cnt.is_contiguous()):
            raise RuntimeError("cnt must be a contiguous int32 CUDA tensor (it is updated in place)")
        CH = int(image_weights.size(0))
        with torch.no_grad():
            # the reference passes `weights` in the colors_precomp slot (rasterize_points.cu:223), so SH
            # evaluation is skipped; the forward's colours are never used
            # (any valid [P,3] float buffer will do for that slot -- means3D avoids an allocation)
            _, _, state, inputs = _forward_impl(means3D, empty, means3D, opacities, scales if scales is not None else empty,
                                                rotations if rotations is not None else empty,
                                                cov3Ds_precomp if cov3Ds_precomp is not None else empty, rs,
                                                render=False)
            if state.P == 0 or state.num_rendered == 0:
                return
            (m3, sh_, cp_, op_, sc_, ro_, cv_) = inputs
            with torch.cuda.device(device):
                keep = []
                s = _make_settings(rs, 0, device, keep)
                c = _make_cloud(state.P, m3, op_, sh_, cp_, sc_, ro_, cv_)
                iw = _f32c(image_weights, device)
                st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
                _lib.check(lib.gsr_apply_weights(C.byref(s), C.byref(c), state.num_rendered, _ptr(state.geom),
                                                 state.geom.numel(), _ptr(state.binning), state.binning.numel(),
                                                 _ptr(state.img), state.img.numel(), _ptr(state.radii), _ptr(iw), CH,
                                                 _ptr(weights), _ptr(cnt), st), "gsr_apply_weights")


# ---- instrumentation for parity tests (not part of the reference API) ---------------------------------------
def forward_state_views(state: _ForwardState):
    """Decode the opaque workspaces of a forward into torch tensors (views onto the workspace memory)."""
    lib = _lib.load()
    P, R, W, H = state.P, state.num_rendered, state.W, state.H
    cap = state.cap
    out = {}

    def view(ptr, base: torch.Tensor, numel, dtype):
        off = ptr - base.data_ptr()
        nbytes = numel * torch.empty(0, dtype=dtype).element_size()
        return base[off:off + nbytes].view(dtype)

    if P == 0:
        dev = state.radii.device
        e = lambda dt, *shape: torch.empty(*shape, dtype=dt, device=dev)
        out.update(records=e(torch.float32, 0, 12), tiles_touched=e(torch.int32, 0), clamped=e(torch.uint8, 0),
                   depth_order=e(torch.int32, 0), point_list=e(torch.int32, 0), tile_keys=e(torch.int32, 0),
                   final_T=e(torch.float32, H, W), n_contrib=e(torch.int32, H, W),
                   ranges=torch.zeros(((W + 15) // 16) * ((H + 15) // 16), 2, dtype=torch.int32, device=dev))
        return out
    gv = _lib.GeometryView()
    _lib.check(lib.gsr_view_geometry(_ptr(state.geom), P, C.byref(gv)), "gsr_view_geometry")
    out["records"] = view(gv.records, state.geom, P * 12, torch.float32).view(P, 12)
    out["tiles_touched"] = view(gv.tiles_touched, state.geom, P, torch.int32)
    out["clamped"] = view(gv.clamped, state.geom, P, torch.uint8)
    out["depth_order"] = view(gv.depth_order, state.geom, P, torch.int32)
    iv = _lib.ImageView()
    _lib.check(lib.gsr_view_image(_ptr(state.img), W, H, C.byref(iv)), "gsr_view_image")
    ntile = ((W + 15) // 16) * ((H + 15) // 16)
    out["final_T"] = view(iv.final_T, state.img, W * H, torch.float32).view(H, W)
    out["n_contrib"] = view(iv.n_contrib, state.img, W * H, torch.int32).view(H, W)
    out["ranges"] = view(iv.ranges, state.img, ntile * 2, torch.int32).view(ntile, 2)
    if R > 0:
        bv = _lib.BinningView()
        _lib.check(lib.gsr_view_binning(_ptr(state.binning), P, cap, W, H, C.byref(bv)), "gsr_view_binning")
        out["point_list"] = view(bv.point_list, state.binning, R, torch.int32)
        out["tile_keys"] = view(bv.tile_keys, state.binning, R, torch.int16 if bv.tile_key_bytes == 2 else torch.int32)
    else:
        out["point_list"] = torch.empty(0, dtype=torch.int32, device=state.geom.device)
        out["tile_keys"] = torch.empty(0, dtype=torch.int32, device=state.geom.device)
    return out
