"""CPU checks of the depth-image gradient (gsr_backward_depth / GaussianRasterizer(..., depth_grad=True)).

The depth image D = sum_i d_i * alpha_i * T_i is blended exactly like a colour channel with colour d_i (the view depth
of Gaussian i) and no background. So on the CPU oracle, which has no depth gradient of its own, the depth loss
sum G_D * D is the colour loss sum (G_D, 0, 0) * C of the same scene rendered with colors_precomp = (d_i, 0, 0) and
bg = 0, plus the chain from d_i to the mean: d_i = V[2] x + V[6] y + V[10] z + V[14] (column-major view matrix).
`depth_truth` builds the gradient of  sum G_C * C + sum G_D * D  that way; the GPU tests (test_depth_grad_gpu.py)
compare the kernels against it. Here it is pinned by (1) the identity itself and (2) central finite differences of the
fp64 oracle's forward."""
import ctypes as C

import numpy as np

from gaussianeditor_b200 import _lib, synth
from oracle import cpu_oracle
from util import axis_camera, rel_l2

GRAD_KEYS = ("dmean2D", "dconic", "dopacity", "dcolor", "dmean3D", "dcov3D", "dsh", "dscale", "drot")


def depth_colors(depths):
    """colors_precomp [P,3] = (d_i, 0, 0) in float32 (what the oracle reads)."""
    d = np.asarray(depths, np.float32)
    return np.ascontiguousarray(np.stack([d, np.zeros_like(d), np.zeros_like(d)], 1))


def depth_truth(cloud, cam, bg, G_C, G_D, f32=False, colors_precomp=None, cov3D_precomp=None):
    """Gradient of  sum G_C * C + sum G_D * D  on the CPU oracle (f32=False: fp64 arithmetic), from the depth-as-colour
    identity. Returns the oracle's gradient dict (rasterize_points.cu:120-128 names) and the forward of the real scene."""
    kw = dict(f32=f32, colors_precomp=colors_precomp)
    if cov3D_precomp is not None:
        kw.update(scales=None, rotations=None, cov3D_precomp=cov3D_precomp)
    f = cpu_oracle.forward_from(cloud, cam, bg, **kw)
    g = f.backward(G_C)
    kw["colors_precomp"] = depth_colors(f.depths)
    fd = cpu_oracle.forward_from(cloud, cam, (0.0, 0.0, 0.0), **kw)
    gd = fd.backward(np.stack([G_D, np.zeros_like(G_D), np.zeros_like(G_D)]))
    fd.close()
    out = {k: g[k] + gd[k] for k in GRAD_KEYS if k not in ("dcolor", "dsh")}
    out["dcolor"], out["dsh"] = g["dcolor"], g["dsh"]
    out["ddepth"] = gd["dcolor"][:, 0]                                   # dL/dd_i = sum alpha_i T_i G_D
    out["dmean3D"] = out["dmean3D"] + out["ddepth"][:, None] * np.asarray(cam.viewmatrix, np.float64)[:3, 2][None, :]
    return out, f


def fd_scene(seed=0, P=200, W=64, H=48):
    """A small scene on which the pipeline is as smooth as it gets: every Gaussian fully in front of axis_camera(W, H)
    and well inside the frame, opacities in [0.2, 0.6] (no pixel comes near the T < 1e-4 stop), non-negative SH
    colours (no clamping), footprints of a few pixels."""
    rng = np.random.default_rng(seed)
    tany = np.tan(np.radians(25.0))
    tanx = tany * W / H
    z = rng.uniform(2.0, 6.0, P)
    ndc = rng.uniform(-0.8, 0.8, (P, 2))
    cam_xyz = np.stack([ndc[:, 0] * tanx * z, ndc[:, 1] * tany * z, z], 1)
    xyz = np.stack([-cam_xyz[:, 0], -cam_xyz[:, 1], cam_xyz[:, 2] - 3.5], 1).astype(np.float32)
    scales = (rng.uniform(0.04, 0.1, (P, 3)) * z[:, None] / 3.0).astype(np.float32)
    q = rng.standard_normal((P, 4))
    rot = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    opac = rng.uniform(0.2, 0.6, (P, 1)).astype(np.float32)
    shs = np.zeros((P, 4, 3), np.float32)
    shs[:, 0] = (rng.uniform(0.3, 0.7, (P, 3)) - 0.5) / 0.28209479177387814
    shs[:, 1:] = rng.standard_normal((P, 3, 3)) * 0.05
    return synth.Cloud(xyz, scales, rot, opac, shs, 1), axis_camera(W, H)


def test_depth_image_is_colour_channel_0_of_the_depth_coloured_scene():
    """fp32 oracle: with colors_precomp = (d_i, 0, 0) and bg = 0, colour channel 0 equals the depth image bit for bit --
    both are  sum x * alpha * T  over the same splats in the same order, and + T_final * 0 adds an exact zero."""
    from util import adversarial_scene
    for cloud, cam in (fd_scene(1), (adversarial_scene()[0], axis_camera(333, 201))):
        f = cpu_oracle.forward_from(cloud, cam, (0.0, 0.0, 0.0))
        fc = cpu_oracle.forward_from(cloud, cam, (0.0, 0.0, 0.0), colors_precomp=depth_colors(f.depths))
        assert np.array_equal(fc.radii, f.radii) and np.array_equal(fc.n_contrib, f.n_contrib)
        assert np.array_equal(fc.color[0], f.depth[0])
        assert np.array_equal(fc.color[1:], np.zeros_like(fc.color[1:]))
        assert float(np.abs(f.depth).max()) > 1.0
        f.close(); fc.close()


# Central differences of the fp64 forward against depth_truth. The analytic gradient (the reference's, for every
# parameter) ignores the motion of the pipeline's edges -- the alpha = 1/255 contour, the 3-sigma tile rectangle, two
# overlapping splats trading places in depth -- while a finite difference integrates any edge it crosses: on this scene
# steps of 2^-10 .. 2^-15 put a handful of Gaussians across an edge and leave rel. L2 errors of 10-40 % (both in the
# colour-only and in the depth-only loss). The steps below cross none, so the difference is the derivative to rounding
# (the fp64 oracle reads d_i as float32 colours). Calibrated on this scene (seed 0): rel. L2 of the whole array
# 3.5e-8 (dopacity) and 3.8e-8 (dmean3D); the depth-only loss: 3.5e-8 and 3.8e-8.
FD_STEP = {"opacities": 2.0 ** -14, "means3D": 2.0 ** -17}
FD_TOL = 1e-6


def _fd_loss(cloud, cam, bg, G_C, G_D, **over):
    c = synth.Cloud(over.get("means3D", cloud.means3D), cloud.scales, cloud.rotations,
                    over.get("opacities", cloud.opacities), cloud.shs, cloud.sh_degree)
    f = cpu_oracle.forward_from(c, cam, bg, f32=False)
    v = float((f.color * G_C).sum() + (f.depth[0] * G_D).sum())
    f.close()
    return v


def _finite_differences(cloud, cam, bg, G_C, G_D, name, h):
    arr = np.ascontiguousarray(getattr(cloud, name), np.float32)
    fd = np.zeros(arr.shape, np.float64)
    for idx in np.ndindex(arr.shape):
        ap, am = arr.copy(), arr.copy()
        ap[idx] += h; am[idx] -= h
        fd[idx] = (_fd_loss(cloud, cam, bg, G_C, G_D, **{name: ap}) -
                   _fd_loss(cloud, cam, bg, G_C, G_D, **{name: am})) / float(ap[idx] - am[idx])
    return fd


def test_depth_truth_matches_finite_differences_of_the_fp64_oracle():
    cloud, cam = fd_scene(0)
    H, W = cam.image_height, cam.image_width
    rng = np.random.default_rng(7)
    bg = (0.2, 0.1, 0.3)
    G_C = rng.standard_normal((3, H, W)).astype(np.float32)
    G_D = rng.standard_normal((H, W)).astype(np.float32)
    want, f = depth_truth(cloud, cam, bg, G_C, G_D)
    assert f.final_T.min() > 1e-3 and not f.clamped.any() and (f.radii > 0).all()
    f.close()
    got = {}
    for name, key in (("opacities", "dopacity"), ("means3D", "dmean3D")):
        fd = _finite_differences(cloud, cam, bg, G_C, G_D, name, np.float32(FD_STEP[name]))
        err = rel_l2(want[key].reshape(fd.shape), fd)
        got[name] = err
        assert err <= FD_TOL, (name, err)
    # the depth term alone (G_C = 0) is a large part of the loss, not a rounding error of it
    zero = np.zeros_like(G_C)
    wd, f = depth_truth(cloud, cam, bg, zero, G_D)
    f.close()
    for name, key in (("opacities", "dopacity"), ("means3D", "dmean3D")):
        fd = _finite_differences(cloud, cam, bg, zero, G_D, name, np.float32(FD_STEP[name]))
        assert np.linalg.norm(fd) > 0.1 * np.linalg.norm(want[key])
        err = rel_l2(wd[key].reshape(fd.shape), fd)
        assert err <= FD_TOL, ("depth only", name, err)
        got["depth-only " + name] = err
    print("rel. L2 against finite differences:", got)


def test_depth_entry_points_validate_before_touching_the_device():
    """gsr_backward_depth / gsr_backward_raw_depth refuse a null depth gradient up front (dummy device pointers are
    never dereferenced)."""
    lib = _lib.load()
    dummy = C.c_void_p(256)
    s = _lib.Settings(64, 64, 1.0, 1.0, 1.0, 0, 1, 0, 0, dummy, dummy, dummy, dummy)
    cloud = _lib.Cloud(10, dummy, dummy, dummy, None, dummy, dummy, None)
    gr = _lib.Grads(*([dummy] * 8))
    cam = _lib.CameraGrads(dummy, dummy, dummy, dummy, 1 << 20)
    for camera in (None, C.byref(cam)):
        rc = lib.gsr_backward_depth(C.byref(s), C.byref(cloud), 100, dummy, 1 << 20, dummy, 1 << 20, dummy, 1 << 20,
                                    dummy, dummy, None, None, dummy, 1 << 20, C.byref(gr), camera, None)
        assert rc == -1 and b"dL_dout_depth is null" in lib.gsr_last_error()
    raw = _lib.RawCloud(10, dummy, dummy, dummy, dummy, dummy, dummy)
    rgr = _lib.RawGrads(*([dummy] * 7))
    rc = lib.gsr_backward_raw_depth(C.byref(s), C.byref(raw), 100, dummy, 1 << 20, dummy, 1 << 20, dummy, 1 << 20,
                                    dummy, dummy, None, dummy, 1 << 20, C.byref(rgr), None)
    assert rc == -1 and b"dL_dout_depth is null" in lib.gsr_last_error()
    # the other argument checks still apply with a depth gradient: both SHs and colours missing
    bad = _lib.Cloud(10, dummy, dummy, None, None, dummy, dummy, None)
    rc = lib.gsr_backward_depth(C.byref(s), C.byref(bad), 100, dummy, 1 << 20, dummy, 1 << 20, dummy, 1 << 20,
                                dummy, dummy, None, dummy, dummy, 1 << 20, C.byref(gr), None, None)
    assert rc == -1 and b"excatly one of either SHs or precomputed colors" in lib.gsr_last_error()
