"""Shared helpers of the test-suite."""
import contextlib
import math

import numpy as np
import torch

from gaussianeditor_b200 import _lib, synth
from gaussianeditor_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer

# The kernel options and their compiled defaults (struct Options, csrc/common.cuh; tests/test_abi_and_host.py checks
# that the two agree). A test that changes an option goes through kernel_options() so that no later test runs on a
# variant it did not ask for.
OPTION_DEFAULTS = dict(render_fwd_variant=3, render_bwd_variant=14, preprocess_variant=1, profile=0, tile_key_bits=16,
                       binning_variant=1, depth_sort_variant=0)


def get_option(name):
    v = int(_lib.load().gsr_get_option(name.encode()))
    assert v != -1, f"unknown kernel option {name}"
    return v


@contextlib.contextmanager
def kernel_options(**opts):
    """Set kernel options (gsr_set_option) for the body of a `with` block; restores the previous values on exit."""
    saved = {k: get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            _lib.set_option(k, v)
        yield
    finally:
        for k, v in saved.items():
            _lib.set_option(k, v)


def settings_from(cam: synth.Camera, bg, sh_degree, device, scale_modifier=1.0, debug=False):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
    return GaussianRasterizationSettings(
        image_height=cam.image_height, image_width=cam.image_width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
        bg=t(np.asarray(bg, np.float32)), scale_modifier=scale_modifier, viewmatrix=t(cam.viewmatrix),
        projmatrix=t(cam.projmatrix), sh_degree=sh_degree, campos=t(cam.campos), prefiltered=False, debug=debug)


def cloud_tensors(cloud: synth.Cloud, device, requires_grad=False):
    t = lambda a: torch.from_numpy(a).to(device).requires_grad_(requires_grad)
    return dict(means3D=t(cloud.means3D), opacities=t(cloud.opacities), shs=t(cloud.shs), scales=t(cloud.scales),
                rotations=t(cloud.rotations))


def run_ours(cloud, cam, bg=(0, 0, 0), dL=None, colors_precomp=None, scale_modifier=1.0, device="cuda"):
    """Forward (+ backward if dL is given) through the public GaussianRasterizer API. Returns dict."""
    from gaussianeditor_b200.rasterizer import _RasterizeGaussians, forward_state_views
    ct = cloud_tensors(cloud, device, requires_grad=dL is not None)
    rs = settings_from(cam, bg, cloud.sh_degree, device, scale_modifier)
    rast = GaussianRasterizer(rs)
    means2D = torch.zeros_like(ct["means3D"], requires_grad=dL is not None)
    kw = dict(means3D=ct["means3D"], means2D=means2D, opacities=ct["opacities"], scales=ct["scales"],
              rotations=ct["rotations"])
    cp = None
    if colors_precomp is not None:
        cp = torch.from_numpy(colors_precomp).to(device).requires_grad_(dL is not None)
        kw["colors_precomp"] = cp
    else:
        kw["shs"] = ct["shs"]
    color, radii, depth = rast(**kw)
    state = _RasterizeGaussians.last_state
    out = dict(color=color.detach(), radii=radii, depth=depth.detach(), R=state.num_rendered,
               views=forward_state_views(state), state=state)
    if dL is not None:
        (color * torch.from_numpy(dL).to(device)).sum().backward()
        out["grads"] = dict(dmean3D=ct["means3D"].grad, dmean2D=means2D.grad, dopacity=ct["opacities"].grad,
                            dscale=ct["scales"].grad, drot=ct["rotations"].grad,
                            dsh=None if cp is not None else ct["shs"].grad, dcolor=None if cp is None else cp.grad)
    return out


def axis_camera(W, H):
    """Camera at (0, 0, -3.5) looking down +z with 50 degrees vertical field of view. Its rotation is diag(-1, -1, 1),
    so the view depth of a point is exactly z + 3.5 in float32: Gaussians with equal z have bit-equal depths."""
    return synth.look_at_camera((0, 0, -3.5), (0, 0, 0), (0, -1, 0), W, H, fovy_deg=50.0)


def adversarial_scene(seed=0, aspect=333 / 201):
    """A scene of the splats where rasterizer kernels go wrong, on top of an ordinary bulk (for axis_camera()).
    Returns (Cloud, {class: Gaussian indices}). Classes: needles (axis ratio 1e2..1e3, up to hundreds of pixels
    long), huge splats just in front of the camera, sub-pixel splats, centres off-screen (|ndc| 1.16..1.6) whose
    rectangle reaches the frame, groups with bit-equal depths, dense stacks that saturate the middle of a tile (the
    T < 1e-4 stop), colours driven negative by the SH DC term (clamping), and opacities at 1/255 * (1 +- 1e-3) or in
    [0.99, 1]."""
    rng = np.random.default_rng(seed)
    tany = math.tan(math.radians(25.0))
    tanx = tany * aspect
    parts, cls = [], {}

    def add(name, n, z, ndc, scales):
        """n Gaussians at camera depth z and normalised device coordinates ndc [n, 2]."""
        start = sum(len(p[0]) for p in parts)
        cam = np.stack([ndc[:, 0] * tanx * z, ndc[:, 1] * tany * z, z], 1)
        parts.append((cam, np.broadcast_to(scales, (n, 3))))
        cls[name] = np.arange(start, start + n)

    u = lambda lo, hi, *s: rng.uniform(lo, hi, s)
    add("bulk", 3000, u(2, 8, 3000), u(-1, 1, 3000, 2), np.exp(rng.normal(math.log(0.03), 0.5, (3000, 3))))
    major = u(0.2, 1.5, 200)
    minor = major / 10.0 ** u(2, 3, 200)
    add("needle", 200, u(3, 6, 200), u(-0.9, 0.9, 200, 2), np.stack([major, minor, minor], 1))
    add("huge", 6, u(0.6, 1.2, 6), u(-0.3, 0.3, 6, 2), u(0.2, 0.6, 6, 3))
    add("subpixel", 300, u(3, 8, 300), u(-1, 1, 300, 2), u(1e-4, 1e-3, 300, 3))
    ndc = u(-1, 1, 150, 2)
    axis = rng.integers(0, 2, 150)
    ndc[np.arange(150), axis] = rng.choice([-1.0, 1.0], 150) * u(1.16, 1.6, 150)
    add("offscreen", 150, u(2, 5, 150), ndc, u(0.3, 0.8, 150, 3))
    # 20 groups of 10 overlapping Gaussians; a group shares one world z -> one depth
    zg = np.repeat(u(2, 7, 20).astype(np.float32), 10)
    add("equal_depth", 200, zg, np.repeat(u(-0.8, 0.8, 20, 2), 10, 0) + u(-0.05, 0.05, 200, 2),
        u(0.02, 0.05, 200, 3))
    # 5 stacks of 40 opaque splats centred inside a tile
    add("stack", 200, u(2, 3, 200), np.repeat(u(-0.7, 0.7, 5, 2), 40, 0), np.repeat(u(0.02, 0.04, 200, 1), 3, 1))
    cam = np.concatenate([p[0] for p in parts])
    scales = np.concatenate([p[1] for p in parts]).astype(np.float32)
    P = len(cam)
    # camera -> world: x_w = -x_c, y_w = -y_c, z_w = z_c - 3.5 (the equal-depth groups keep their float32 z_c)
    xyz = np.stack([-cam[:, 0], -cam[:, 1], cam[:, 2] - 3.5], 1).astype(np.float32)
    xyz[cls["equal_depth"], 2] = zg - np.float32(3.5)
    q = rng.standard_normal((P, 4))
    rot = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    opac = 1.0 / (1.0 + np.exp(-rng.normal(0.0, 2.0, P)))
    opac[cls["huge"]] = u(0.05, 0.3, 6)
    opac[cls["stack"]] = u(0.9, 0.99, 200)
    perm = rng.permutation(P)
    cls["opacity_1_255"] = perm[:150]
    opac[cls["opacity_1_255"]] = (1.0 + rng.choice([-1e-3, 1e-3], 150)) / 255.0
    cls["opacity_high"] = perm[150:300]
    opac[cls["opacity_high"]] = u(0.99, 1.0, 150)
    shs = np.zeros((P, 16, 3), np.float32)
    shs[:, 0, :] = (u(0, 1, P, 3) - 0.5) / 0.28209479177387814
    for ell, (a, b) in enumerate([(1, 4), (4, 9), (9, 16)], 1):
        shs[:, a:b, :] = rng.standard_normal((P, b - a, 3)) * (0.15 / (1 + ell))
    cls["negative_colour"] = perm[300:700]
    shs[cls["negative_colour"], 0, rng.integers(0, 3, 400)] = -3.0
    cloud = synth.Cloud(xyz, scales, rot, opac.astype(np.float32)[:, None], shs, 3)
    return cloud, cls


def bin_reference(means2D, radii, depths, W, H):
    """The reference's binning (duplicateWithKeys + stable radix sort + identifyTileRanges) restated in numpy, from
    the per-Gaussian projected centres, radii and fp32 view depths. Returns tiles_touched [P] (uint32), R,
    ranges [ntile, 2] (uint32; (0, 0) for an empty tile) and point_list [R] (uint32): every (Gaussian, tile) instance
    of a Gaussian with radius > 0, ordered by (tile id, depth bits, Gaussian index)."""
    f = np.float32
    gx, gy = (W + 15) // 16, (H + 15) // 16
    radii = np.asarray(radii).astype(np.int64)
    idx = np.flatnonzero(radii > 0)
    px, py = (np.asarray(means2D, f)[idx, k] for k in (0, 1))
    r = radii[idx].astype(f)

    def cell(v, g):  # (int)(v / 16) truncates toward zero, then clamped to [0, g] (tile_binning.cu tile_rect)
        return np.clip(np.trunc(v / f(16)).astype(np.int64), 0, g)
    # float32, left to right as the kernel evaluates it: (px - r) / 16 and (((px + r) + 16) - 1) / 16
    x0, y0 = cell(px - r, gx), cell(py - r, gy)
    x1, y1 = cell(((px + r) + f(16)) - f(1), gx), cell(((py + r) + f(16)) - f(1), gy)
    w = x1 - x0
    n = w * (y1 - y0)
    tiles_touched = np.zeros(len(radii), np.uint32)
    tiles_touched[idx] = n
    R = int(n.sum())
    owner = np.repeat(np.arange(len(idx)), n)                       # emission order: by Gaussian index
    k = np.arange(R) - np.repeat(np.cumsum(n) - n, n)               # position inside the Gaussian's rectangle
    wk = np.maximum(np.repeat(w, n), 1)
    tile = (np.repeat(y0, n) + k // wk) * gx + np.repeat(x0, n) + k % wk
    dbits = np.ascontiguousarray(np.asarray(depths, f)[idx]).view(np.uint32).astype(np.uint64)
    key = (tile.astype(np.uint64) << np.uint64(32)) | dbits[owner]
    order = np.argsort(key, kind="stable")                          # == np.lexsort((index, depth_bits, tile))
    point_list = idx[owner[order]].astype(np.uint32)
    cnt = np.bincount(tile, minlength=gx * gy).astype(np.int64)
    end = np.cumsum(cnt)
    ranges = np.where((cnt > 0)[:, None], np.stack([end - cnt, end], 1), 0).astype(np.uint32)
    return dict(tiles_touched=tiles_touched, R=R, ranges=ranges, point_list=point_list)


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
