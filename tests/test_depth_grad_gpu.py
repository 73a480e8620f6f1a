"""GPU tests of the depth-image gradient: GaussianRasterizer(..., depth_grad=True) -> gsr_backward_depth /
gsr_backward_raw_depth -> the DEPTH instantiations of render_bwd and the depth term of preprocess_bwd.

  1. own-path identity: a depth loss equals a colour loss on colors_precomp = (d_i, 0, 0) built in PyTorch (autograd
     then supplies the chain d_i -> means3D / viewmatrix), bg = 0;
  2. every render_bwd variant, per Gaussian, against the fp64 truth of test_depth_grad_cpu.depth_truth on
     util.adversarial_scene (SH, precomputed colours, precomputed covariance) with a signed colour + depth loss;
  3. no change without the flag (bit for bit where the float atomics have a fixed order), none with a zero depth
     gradient;
  4. alpha + camera + depth in one call, the fused-activation path, render();
  5. shapes: P = 0, everything culled, one tile, frames that are not multiples of 16.
Every test runs with the kernel options at their compiled defaults unless it sets one through util.kernel_options."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from gaussianeditor_b200 import synth
from test_depth_grad_cpu import depth_truth
from test_shapes_and_variants_gpu import (BG, BWD_VARIANTS, DIRECT, TOL_FP64, TOL_VARIANT, failing_rows, row_terms,
                                          signed_dL)
from util import OPTION_DEFAULTS, adversarial_scene, axis_camera, get_option, kernel_options, rel_l2, settings_from

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(autouse=True, scope="module")
def options_at_compiled_defaults():
    assert {k: get_option(k) for k in OPTION_DEFAULTS} == OPTION_DEFAULTS
    yield
    assert {k: get_option(k) for k in OPTION_DEFAULTS} == OPTION_DEFAULTS


def _t(a, grad=False):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV).requires_grad_(grad)


def render(cloud, cam, bg, G_C=None, G_D=None, G_A=None, depth_grad=False, camera_grad=False, colors_precomp=None,
           cov3D_precomp=None):
    """Forward + backward of  sum G_C*C + sum G_D*D (+ sum G_A*alpha)  through the public API. colors_precomp may be a
    numpy array or a callable (means3D, viewmatrix) -> tensor (built inside the graph). Returns (outputs, grads)."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    m3 = _t(cloud.means3D, True)
    m2 = torch.zeros_like(m3, requires_grad=True)
    op = _t(cloud.opacities, True)
    rs = settings_from(cam, bg, cloud.sh_degree, DEV)
    leaves = dict(means3D=m3, means2D=m2, opacities=op)
    if camera_grad:
        cams = {k: getattr(rs, k).clone().requires_grad_(True) for k in ("viewmatrix", "projmatrix", "campos")}
        rs = rs._replace(**cams)
        leaves.update(cams)
    kw = dict(means3D=m3, means2D=m2, opacities=op)
    if cov3D_precomp is not None:
        kw["cov3D_precomp"] = leaves["cov3D"] = _t(cov3D_precomp, True)
    else:
        kw["scales"] = leaves["scales"] = _t(cloud.scales, True)
        kw["rotations"] = leaves["rotations"] = _t(cloud.rotations, True)
    if callable(colors_precomp):
        kw["colors_precomp"] = colors_precomp(m3, rs.viewmatrix)
    elif colors_precomp is not None:
        kw["colors_precomp"] = leaves["colors"] = _t(colors_precomp, True)
    else:
        kw["shs"] = leaves["shs"] = _t(cloud.shs, True)
    out = GaussianRasterizer(rs, return_alpha=G_A is not None, camera_grad=camera_grad, depth_grad=depth_grad)(**kw)
    loss = 0.0
    if G_C is not None:
        loss = loss + (out[0] * _t(G_C)).sum()
    if G_D is not None:
        loss = loss + (out[2][0] * _t(G_D)).sum()
    if G_A is not None:
        loss = loss + (out[3][0] * _t(G_A)).sum()
    loss.backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)).detach() for k, v in leaves.items()}
    return out, grads


def depth_as_colour(means3D, view):
    """(d_i, 0, 0) with d_i = means3D @ V[:3, 2] + V[3, 2], the view depth, in PyTorch."""
    d = means3D @ view[:3, 2] + view[3, 2]
    z = torch.zeros_like(d)
    return torch.stack([d, z, z], 1)


def _assert_close(ga, gb, keys, tol):
    for k in keys:
        e = rel_l2(ga[k].cpu().numpy(), gb[k].cpu().numpy())
        assert e <= tol, (k, e)


# ---- 1. own-path identity ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("camera_grad", [False, True])
def test_depth_loss_equals_colour_loss_on_depth_coloured_splats(camera_grad):
    """Run A: sum G_D*D with depth_grad on the SH path. Run B: the same scene with colors_precomp = (d_i, 0, 0) built in
    PyTorch from means3D and the view matrix, bg = 0, loss sum G_D*C_0. Same bound as the alpha identity (2e-5). With
    camera gradients all three camera arrays are compared: the view matrix receives the d_i chain on top of what
    mean2D / conic pass on; projmatrix (through mean2D) gets no direct depth term, campos (SH colours only) nothing."""
    cloud, _ = synth.make_config("c3", P=40_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 333, 201, 61.0)[2]
    H, W = cam.image_height, cam.image_width
    G = np.random.default_rng(29).standard_normal((H, W)).astype(np.float32)
    out_a, ga = render(cloud, cam, (0.0, 0.0, 0.0), G_D=G, depth_grad=True, camera_grad=camera_grad)
    G3 = np.stack([G, np.zeros_like(G), np.zeros_like(G)])
    out_b, gb = render(cloud, cam, (0.0, 0.0, 0.0), G_C=G3, colors_precomp=depth_as_colour, camera_grad=camera_grad)
    assert rel_l2(out_b[0][0].detach().cpu().numpy(), out_a[2][0].detach().cpu().numpy()) <= 1e-6
    keys = ["means3D", "means2D", "opacities", "scales", "rotations"]
    if camera_grad:
        keys += ["viewmatrix", "projmatrix", "campos"]
        assert float(ga["campos"].abs().max()) == 0.0 and float(ga["viewmatrix"].abs().max()) > 0
    assert float(ga["means3D"].abs().max()) > 0 and float(ga["means2D"].abs().max()) > 0
    _assert_close(ga, gb, keys, 2e-5)


# ---- 2. every variant against the fp64 truth -------------------------------------------------------------------------
KEYS = {"sh": ("dmean2D", "dopacity", "dsh", "dmean3D", "dscale", "drot"),
        "colors": ("dmean2D", "dopacity", "dcolor", "dmean3D", "dscale", "drot"),
        "cov3D": ("dmean2D", "dopacity", "dsh", "dmean3D", "dcov3D")}
OURS = dict(dmean2D="means2D", dopacity="opacities", dsh="shs", dcolor="colors", dmean3D="means3D", dscale="scales",
            drot="rotations", dcov3D="cov3D")


def _ours(g, k):
    x = g[OURS[k]]
    return x[:, :2] if k == "dmean2D" else x


def _ratio(terms, tol):
    d, ferr, n, nmax = terms
    a, b, c = tol
    return float(np.max(d / (a * ferr + b * n + c * nmax)))


@pytest.mark.parametrize("path", ["sh", "colors", "cov3D"])
def test_every_variant_against_fp64_depth_truth(path):
    """util.adversarial_scene, signed colour loss (zeroed block, one channel x 10^3) + signed depth loss, nonzero
    background. Per Gaussian with test_shapes_and_variants_gpu's bounds: against the fp64 truth (TOL_FP64, at most
    max(2, 1e-4 V) rows off -- alpha on the 1/255 or T contour decided differently with and without FMA contraction) and
    against variant 0 (TOL_VARIANT, no row off). The worst ratios (left side / right side) are printed; the bounds are
    the existing ones, not re-calibrated. Worst observed on a B200 (1000 W power limit), two runs, all three paths and 15
    variants: fp64 direct 0.73, fp64 chain 0.97 (precomputed colours), variant 0 direct 0.49, variant 0 chain 0.69."""
    W, H = 333, 201
    cloud, _ = adversarial_scene()
    cam = axis_camera(W, H)
    P = cloud.means3D.shape[0]
    G_C = signed_dL(H, W, seed=11)
    G_D = np.random.default_rng(13).standard_normal((H, W)).astype(np.float32)
    G_D[H // 2:, :W // 3] = 0.0
    cp = cov = None
    if path == "colors":
        cp = np.random.default_rng(5).uniform(-0.2, 1.2, (P, 3)).astype(np.float32)
    if path == "cov3D":
        from oracle import cpu_oracle
        f = cpu_oracle.forward_from(cloud, cam, BG)
        cov = np.ascontiguousarray(f.cov3D, np.float32)
        f.close()
    e, f = depth_truth(cloud, cam, BG, G_C, G_D, f32=False, colors_precomp=cp, cov3D_precomp=cov)
    f.close()
    fo, f = depth_truth(cloud, cam, BG, G_C, G_D, f32=True, colors_precomp=cp, cov3D_precomp=cov)
    f.close()
    outs = {}
    for v in BWD_VARIANTS:
        with kernel_options(render_bwd_variant=v):
            outs[v] = render(cloud, cam, BG, G_C=G_C, G_D=G_D, depth_grad=True, colors_precomp=cp, cov3D_precomp=cov)
    V = int((outs[14][0][1] > 0).sum())
    allowed = max(2, int(1e-4 * V))
    worst = {}
    for v in BWD_VARIANTS:
        g = outs[v][1]
        for k in KEYS[path]:
            ek, fk = e[k], fo[k]
            if k == "dmean2D":
                ek, fk = ek[:, :2], fk[:, :2]
            grp = "direct" if k in DIRECT else "chain"
            t = row_terms(_ours(g, k), ek, ek, fk)
            bad = failing_rows(t, TOL_FP64[grp])
            assert len(bad) <= allowed, (v, k, bad[:20])
            ok = np.setdiff1d(np.arange(len(t[0])), bad)
            worst[("fp64", grp)] = max(worst.get(("fp64", grp), 0.0), _ratio([x[ok] if np.ndim(x) else x for x in t],
                                                                            TOL_FP64[grp]))
            t0 = row_terms(_ours(g, k), _ours(outs[0][1], k), ek, fk)
            bad0 = failing_rows(t0, TOL_VARIANT[grp])
            assert len(bad0) == 0, (v, k, bad0[:20])
            worst[("variant0", grp)] = max(worst.get(("variant0", grp), 0.0), _ratio(t0, TOL_VARIANT[grp]))
    print(f"{path}: worst ratios {worst}")


# ---- 3. no change without the flag -----------------------------------------------------------------------------------
def one_tile_case():
    """A 16 x 8 frame: one tile whose pixels all lie in the first half-tile warp of the default backward, so each
    Gaussian receives exactly one atomic per accumulator slot and the gradients are bit-reproducible."""
    cloud, _ = adversarial_scene(seed=3, aspect=2.0)
    cam = axis_camera(16, 8)
    rng = np.random.default_rng(17)
    return cloud, cam, rng.standard_normal((3, 8, 16)).astype(np.float32), rng.standard_normal((8, 16)).astype(np.float32)


@pytest.mark.parametrize("camera_grad", [False, True])
def test_without_the_flag_the_depth_loss_changes_nothing(camera_grad):
    cloud, cam, G_C, G_D = one_tile_case()
    _, base = render(cloud, cam, BG, G_C=G_C, camera_grad=camera_grad)
    _, again = render(cloud, cam, BG, G_C=G_C, camera_grad=camera_grad)
    for k in base:
        assert torch.equal(base[k], again[k]), ("the one-tile case is not reproducible", k)
    _, with_d = render(cloud, cam, BG, G_C=G_C, G_D=G_D, camera_grad=camera_grad)
    for k in base:
        assert torch.equal(with_d[k], base[k]), k
    # depth_grad with a zero depth gradient: the same bits (torch.equal: -0 == +0)
    _, zero_d = render(cloud, cam, BG, G_C=G_C, G_D=np.zeros_like(G_D), depth_grad=True, camera_grad=camera_grad)
    for k in base:
        assert torch.equal(zero_d[k], base[k]), k
    # and a nonzero one does change them
    _, nz = render(cloud, cam, BG, G_C=G_C, G_D=G_D, depth_grad=True, camera_grad=camera_grad)
    assert not torch.equal(nz["means3D"], base["means3D"])


def test_zero_depth_gradient_matches_the_plain_backward_at_full_scene():
    """333 x 201 adversarial scene, default variant: depth_grad with G_D = 0 against depth_grad=False, within the
    run-to-run noise of the float atomics. The noise is measured in the same test: two more plain runs. Per array,
    rel. L2 (zero-depth vs plain) <= 3 x the larger rel. L2 of the plain repeats + 1e-7. (A per-row bound does not fit
    here: on the needles of this scene the fp32 cancellation of the 2-D -> 3-D chain turns the order of the atomics
    into rows that differ by more than TOL_VARIANT between any two runs. The one-tile test above, whose atomics have a
    fixed order, shows that the bits are the same.)"""
    W, H = 333, 201
    cloud, _ = adversarial_scene()
    cam = axis_camera(W, H)
    G_C = signed_dL(H, W, seed=11)
    _, a = render(cloud, cam, BG, G_C=G_C)
    repeats = [render(cloud, cam, BG, G_C=G_C)[1] for _ in range(2)]
    _, b = render(cloud, cam, BG, G_C=G_C, G_D=np.zeros((H, W), np.float32), depth_grad=True)
    report = {}
    for k, x in a.items():
        e = x.cpu().numpy()
        noise = max(rel_l2(r[k].cpu().numpy(), e) for r in repeats)
        got = rel_l2(b[k].cpu().numpy(), e)
        report[k] = (got, noise)
        assert got <= 3.0 * noise + 1e-7, (k, got, noise)
    print("rel. L2 (zero depth vs plain, plain vs plain):", report)


# ---- 4. combinations and paths -----------------------------------------------------------------------------------------
def test_alpha_camera_and_depth_in_one_call_is_the_sum_of_the_parts():
    """The backward is linear in the upstream gradients: (colour + alpha + depth) with return_alpha, camera_grad and
    depth_grad in one call == (colour + alpha) without depth_grad + (depth) alone."""
    cloud, _ = synth.make_config("c3", P=20_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 240, 176, 61.0)[5]
    H, W = cam.image_height, cam.image_width
    rng = np.random.default_rng(41)
    G_C = rng.standard_normal((3, H, W)).astype(np.float32)
    G_A = rng.standard_normal((H, W)).astype(np.float32)
    G_D = rng.standard_normal((H, W)).astype(np.float32)
    bg = (0.2, 0.3, 0.4)
    out, g = render(cloud, cam, bg, G_C=G_C, G_A=G_A, G_D=G_D, depth_grad=True, camera_grad=True)
    assert len(out) == 4
    _, g1 = render(cloud, cam, bg, G_C=G_C, G_A=G_A, camera_grad=True)
    _, g2 = render(cloud, cam, bg, G_D=G_D, depth_grad=True, camera_grad=True)
    for k in g:
        assert torch.isfinite(g[k]).all(), k
        assert rel_l2(g[k].cpu().numpy(), (g1[k] + g2[k]).cpu().numpy()) <= 1e-4, (k, rel_l2(g[k].cpu().numpy(), (g1[k] + g2[k]).cpu().numpy()))
    assert float(g2["viewmatrix"].abs().max()) > 0


def test_fused_activations_with_depth_grad_match_pytorch_prologue():
    """forward_raw with depth_grad against the PyTorch-activated path with depth_grad (rel. L2 <= 1e-4, as in
    test_fused_activations_match_pytorch_prologue)."""
    from gaussianeditor_b200.rasterizer import GaussianRasterizer
    from test_parity_gpu import _raw_params
    cloud, _ = synth.make_config("c3", P=20_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 640, 400, 61.0)[1]
    rs = settings_from(cam, (0.3, 0.1, 0.2), cloud.sh_degree, DEV)
    rng = np.random.default_rng(43)
    G_C = _t(rng.uniform(size=(3, cam.image_height, cam.image_width)).astype(np.float32))
    G_D = _t(rng.standard_normal((cam.image_height, cam.image_width)).astype(np.float32))
    rast = GaussianRasterizer(rs, depth_grad=True)
    a = _raw_params(cloud, DEV)
    m2a = torch.zeros_like(a["xyz"], requires_grad=True)
    col_a, rad_a, dep_a = rast(means3D=a["xyz"], means2D=m2a, opacities=torch.sigmoid(a["opacity"]),
                               shs=torch.cat((a["features_dc"], a["features_rest"]), dim=1),
                               scales=torch.exp(a["scaling"]), rotations=torch.nn.functional.normalize(a["rotation"]))
    ((col_a * G_C).sum() + (dep_a[0] * G_D).sum()).backward()
    b = _raw_params(cloud, DEV)
    m2b = torch.zeros_like(b["xyz"], requires_grad=True)
    col_b, rad_b, dep_b = rast.forward_raw(means3D=b["xyz"], means2D=m2b, opacity_logits=b["opacity"],
                                           features_dc=b["features_dc"], features_rest=b["features_rest"],
                                           log_scales=b["scaling"], raw_rotations=b["rotation"])
    ((col_b * G_C).sum() + (dep_b[0] * G_D).sum()).backward()
    same = rad_a == rad_b
    assert float((~same).float().mean()) <= 1e-4
    for k in a:
        ga, gb = a[k].grad, b[k].grad
        assert gb is not None and torch.isfinite(gb).all(), k
        assert rel_l2(gb[same].cpu().numpy(), ga[same].cpu().numpy()) <= 1e-4, k
    assert rel_l2(m2b.grad[same].cpu().numpy(), m2a.grad[same].cpu().numpy()) <= 1e-4
    # the depth term is really in there: without it the xyz gradient differs
    c = _raw_params(cloud, DEV)
    col_c, _, dep_c = GaussianRasterizer(rs).forward_raw(
        means3D=c["xyz"], means2D=torch.zeros_like(c["xyz"]), opacity_logits=c["opacity"], features_dc=c["features_dc"],
        features_rest=c["features_rest"], log_scales=c["scaling"], raw_rotations=c["rotation"])
    ((col_c * G_C).sum() + (dep_c[0] * G_D).sum()).backward()
    assert rel_l2(c["xyz"].grad.cpu().numpy(), b["xyz"].grad.cpu().numpy()) > 1e-2


def _scene_model(cloud):
    """The scene model's attributes render() reads, as raw leaf tensors (scene/gaussian_model.py)."""
    from test_parity_gpu import _raw_params
    r = _raw_params(cloud, torch.device(DEV))
    pc = SimpleNamespace(_xyz=r["xyz"], _opacity=r["opacity"], _features_dc=r["features_dc"],
                         _features_rest=r["features_rest"], _scaling=r["scaling"], _rotation=r["rotation"],
                         active_sh_degree=cloud.sh_degree)
    pc.get_xyz = pc._xyz
    pc.get_opacity = torch.sigmoid(pc._opacity)
    pc.get_scaling = torch.exp(pc._scaling)
    pc.get_rotation = torch.nn.functional.normalize(pc._rotation)
    pc.get_features = torch.cat((pc._features_dc, pc._features_rest), dim=1)
    return pc


@pytest.mark.parametrize("fused", [False, True])
def test_render_passes_depth_grad_through(fused):
    from gaussianeditor_b200.gaussian_renderer import render as gs_render
    cloud, _ = synth.make_config("c3", P=20_000)
    c = synth.ring_cameras(8, 4.5, 15.0, 320, 240, 61.0)[4]
    vcam = SimpleNamespace(image_height=c.image_height, image_width=c.image_width,
                           FoVx=2 * np.arctan(c.tanfovx), FoVy=2 * np.arctan(c.tanfovy),
                           world_view_transform=_t(c.viewmatrix.astype(np.float32)),
                           full_proj_transform=_t(c.projmatrix.astype(np.float32)),
                           camera_center=_t(c.campos.astype(np.float32)))
    pipe = SimpleNamespace(convert_SHs_python=False, compute_cov3D_python=False)
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    G_D = _t(np.random.default_rng(47).standard_normal((c.image_height, c.image_width)).astype(np.float32))
    grads = {}
    for depth_grad in (False, True):
        pc = _scene_model(cloud)
        pkg = gs_render(vcam, pc, pipe, bg, fused_activations=fused, depth_grad=depth_grad)
        (pkg["depth_3dgs"][0] * G_D).sum().backward()
        grads[depth_grad] = (pc._xyz.grad, pkg["viewspace_points"].grad)
    # without the flag a depth-only loss trains nothing, as in the reference; with it it reaches the means and the
    # densification statistics
    for g in grads[False]:
        assert g is None or float(g.abs().max()) == 0.0
    xyz_g, vs_g = grads[True]
    assert torch.isfinite(xyz_g).all() and float(xyz_g.abs().max()) > 0
    assert torch.isfinite(vs_g).all() and float(vs_g[:, :2].abs().max()) > 0
    if fused:   # the fused path against the PyTorch-activated one
        pc = _scene_model(cloud)
        pkg = gs_render(vcam, pc, pipe, bg, fused_activations=False, depth_grad=True)
        (pkg["depth_3dgs"][0] * G_D).sum().backward()
        assert rel_l2(xyz_g.cpu().numpy(), pc._xyz.grad.cpu().numpy()) <= 1e-4


# ---- 5. shapes -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["empty", "all_culled", "one_tile", "333x201", "7x5"])
def test_depth_grad_shapes(case):
    W, H = {"one_tile": (16, 16), "7x5": (7, 5)}.get(case, (333, 201))
    cam = axis_camera(W, H)
    if case == "empty":
        cloud = synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 4), np.float32),
                            np.zeros((0, 1), np.float32), np.zeros((0, 16, 3), np.float32), 3)
    else:
        cloud, _ = adversarial_scene(aspect=W / H)
        if case == "all_culled":
            cloud.means3D[:, 2] = -10.0
    rng = np.random.default_rng(53)
    G_C = rng.standard_normal((3, H, W)).astype(np.float32)
    G_D = rng.standard_normal((H, W)).astype(np.float32)
    cp = np.zeros((0, 3), np.float32) if case == "empty" else None     # an empty SH array has no coefficient count
    out, g = render(cloud, cam, BG, G_C=G_C, G_D=G_D, depth_grad=True, camera_grad=True, colors_precomp=cp)
    vis = out[1] > 0
    for k, x in g.items():
        assert torch.isfinite(x).all(), k
        if k not in ("viewmatrix", "projmatrix", "campos"):
            assert x.shape[0] == cloud.means3D.shape[0], k
            assert float(x[~vis].abs().sum()) == 0.0, k
    if case in ("empty", "all_culled"):
        assert int(vis.sum()) == 0
        for k, x in g.items():
            assert float(x.abs().sum()) == 0.0, k
    else:
        assert int(vis.sum()) > 0 and float(g["means3D"].abs().max()) > 0
