"""Known-answer tests that pin the CPU oracle (oracle/cpu_rasterizer.cpp) WITHOUT a GPU.

The reference ships no tests or golden vectors for this path (SURVEY.md section 4), so the oracle is pinned by
  (i)   closed-form single-Gaussian answers,
  (ii)  hand-computed two-Gaussian compositing incl. the T<1e-4 stop rule,
  (iii) culling edge cases (near plane, zero-area rectangle, partial last tile row),
  (iv)  independent numpy restatements of the reference's own PyTorch helpers
        (gaussiansplatting/utils/sh_utils.py:57-112 eval_sh, utils/general_utils.py:78-110 build_scaling_rotation),
  (v)   fp64 finite differences of every gradient tensor,
  (vi)  (GPU tests) bit-for-bit comparison with the reference's own CUDA build, and the committed golden vectors
        it produced (tests/test_golden.py).
"""
import math

import numpy as np
import pytest

from gaussianeditor_b200 import synth
from oracle import cpu_oracle as O

C0 = 0.28209479177387814


def _cam(W=64, H=48, fovy=50.0, eye=(0, 0, -3.5)):
    return synth.look_at_camera(eye, (0, 0, 0), (0, -1, 0), W, H, fovy_deg=fovy)


def _cloud(xyz, scales, rots, opac, rgb_dc=None, sh=None, deg=0):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    P = xyz.shape[0]
    if sh is None:
        sh = np.zeros((P, 1, 3), np.float32)
        if rgb_dc is not None:
            sh[:, 0, :] = (np.asarray(rgb_dc, np.float32).reshape(-1, 3) - 0.5) / C0
    return synth.Cloud(xyz, np.asarray(scales, np.float32).reshape(-1, 3), np.asarray(rots, np.float32).reshape(-1, 4),
                       np.asarray(opac, np.float32).reshape(-1, 1), np.asarray(sh, np.float32), deg)


def test_single_isotropic_gaussian_closed_form():
    W, H = 64, 48
    cam = _cam(W, H)
    s = 0.05
    cloud = _cloud([[0, 0, 0]], [[s, s, s]], [[1, 0, 0, 0]], [[0.8]], rgb_dc=[[0.9, 0.5, 0.1]])
    f = O.forward_from(cloud, cam, f32=False)
    # projection: the look-at target is the image centre -> pixel ((W-1)/2, (H-1)/2)
    assert np.allclose(f.means2D[0], [(W - 1) / 2, (H - 1) / 2], atol=1e-4)
    assert abs(f.depths[0] - 3.5) < 1e-6
    fy = H / (2 * cam.tanfovy)
    fx = W / (2 * cam.tanfovx)
    var = (fx * s / 3.5) ** 2 + 0.3           # isotropic: cov2D = (f s / z)^2 I + 0.3 I
    assert abs(fx - fy) < 1e-3
    assert np.allclose(f.conic_opacity[0], [1 / var, 0, 1 / var, 0.8], atol=1e-5)
    lam = var                                   # mid + sqrt(max(0.1, 0)) -> mid + sqrt(0.1)
    radius = math.ceil(3 * math.sqrt(lam + math.sqrt(0.1)))
    assert f.radii[0] == radius
    # alpha at a pixel at distance d from the centre: min(0.99, 0.8 exp(-d^2 / (2 var)))
    px, py = 31, 23                             # centre is (31.5, 23.5)
    d2 = 0.5 ** 2 + 0.5 ** 2
    alpha = 0.8 * math.exp(-0.5 * d2 / var)
    assert abs(f.final_T[py, px] - (1 - alpha)) < 1e-6
    assert np.allclose(f.color[:, py, px], np.array([0.9, 0.5, 0.1]) * alpha, atol=1e-6)
    assert abs(f.depth[0, py, px] - 3.5 * alpha) < 1e-5
    assert f.n_contrib[py, px] == 1
    # far corner: alpha < 1/255 -> untouched, T = 1, background shows through
    g = O.forward_from(cloud, cam, bg=(0.25, 0.5, 0.75), f32=False)
    assert g.final_T[0, 0] == 1.0 and np.allclose(g.color[:, 0, 0], [0.25, 0.5, 0.75])


def test_two_gaussians_compositing_and_stop_rule():
    cam = _cam(32, 32)
    s = 0.5  # huge splats: alpha ~ opacity over the centre region
    # front (z=-1 -> view depth 2.5) opaque-ish red, back (z=+1 -> 4.5) green
    cloud = _cloud([[0, 0, 1.0], [0, 0, -1.0]], [[s] * 3, [s] * 3], [[1, 0, 0, 0]] * 2, [[0.9], [0.6]],
                   rgb_dc=[[0, 1, 0], [1, 0, 0]])
    f = O.forward_from(cloud, cam, f32=False)
    tile_list = f.point_list[f.ranges[0, 0]:f.ranges[0, 1]]
    assert list(tile_list[:2]) == [1, 0]                    # sorted front to back: index 1 (depth 2.5) first
    py = px = 16
    co = f.conic_opacity
    def alpha(i):
        dx, dy = f.means2D[i] - np.array([px, py], np.float64)
        p = -0.5 * (co[i, 0] * dx * dx + co[i, 2] * dy * dy) - co[i, 1] * dx * dy
        return min(0.99, co[i, 3] * math.exp(p))
    a1, a0 = alpha(1), alpha(0)
    assert np.allclose(f.color[:, py, px], [a1, (1 - a1) * a0, 0], atol=1e-7)
    assert abs(f.final_T[py, px] - (1 - a1) * (1 - a0)) < 1e-7
    assert abs(f.depth[0, py, px] - (2.5 * a1 + 4.5 * (1 - a1) * a0)) < 1e-6
    assert f.n_contrib[py, px] == 2
    # stop rule: ten opaque layers, alpha clamps at 0.99f = 0.99000000954: after one layer T = 0.00999999046 and
    # the second would give 9.9999981e-05 < 1e-4f, so the pixel stops with exactly ONE blended splat
    n = 10
    xyz = [[0, 0, -1.0 + 0.1 * i] for i in range(n)]
    cl = _cloud(xyz, [[s] * 3] * n, [[1, 0, 0, 0]] * n, [[1.0]] * n, rgb_dc=[[1, 1, 1]] * n)
    g = O.forward_from(cl, cam, f32=False)
    T = g.final_T[py, px]
    k = g.n_contrib[py, px]
    assert T >= 1e-4 and T * (1 - 0.99) < 1e-4               # the next splat would have crossed the threshold
    assert k == 1 and abs(T - (1.0 - float(np.float32(0.99)))) < 1e-12


def test_culling_edge_cases():
    # camera at the origin looking down +z, so view depth == world z exactly; 40 rows -> 3 tile rows, last partial
    cam = synth.look_at_camera((0, 0, 0), (0, 0, 1), (0, -1, 0), 64, 40, fovy_deg=50.0)
    base = dict(scales=[[0.005] * 3] * 4, rots=[[1, 0, 0, 0]] * 4, opac=[[0.5]] * 4, rgb_dc=[[1, 1, 1]] * 4)
    z_edge = np.float32(0.2)
    xyz = [[0, 0, z_edge], [0, 0, np.nextafter(z_edge, np.float32(1))], [0, 0, -5.0], [50.0, 0, 1.0]]
    f = O.forward_from(_cloud(xyz, **base), cam)
    assert f.radii[0] == 0            # depth exactly 0.2 (<= 0.2) is culled (auxiliary.h:154)
    assert f.radii[1] > 0             # just beyond the near plane survives
    assert f.radii[2] == 0            # behind the camera
    assert f.radii[3] == 0 and f.tiles_touched[3] == 0   # projects far outside: zero-area tile rectangle
    assert f.ranges.shape[0] == 4 * 3
    assert f.num_rendered == int(f.tiles_touched.sum())
    vis = O.mark_visible(np.asarray(xyz, np.float32), cam.viewmatrix)
    assert list(vis) == [False, True, False, True]      # markVisible only applies the near-plane test


def _eval_sh_numpy(deg, sh, d):
    """Restatement of gaussiansplatting/utils/sh_utils.py:57-112 (sh [..,C,(deg+1)^2], d [..,3])."""
    C1 = 0.4886025119029199
    C2 = [1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792, 0.5462742152960396]
    C3 = [-0.5900435899266435, 2.890611442640554, -0.4570457994644658, 0.3731763325901154, -0.4570457994644658,
          1.445305721320277, -0.5900435899266435]
    x, y, z = d[..., 0:1], d[..., 1:2], d[..., 2:3]
    r = C0 * sh[..., 0]
    if deg > 0:
        r = r - C1 * y * sh[..., 1] + C1 * z * sh[..., 2] - C1 * x * sh[..., 3]
        if deg > 1:
            xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
            r = (r + C2[0] * xy * sh[..., 4] + C2[1] * yz * sh[..., 5] + C2[2] * (2.0 * zz - xx - yy) * sh[..., 6] +
                 C2[3] * xz * sh[..., 7] + C2[4] * (xx - yy) * sh[..., 8])
            if deg > 2:
                r = (r + C3[0] * y * (3 * xx - yy) * sh[..., 9] + C3[1] * xy * z * sh[..., 10] +
                     C3[2] * y * (4 * zz - xx - yy) * sh[..., 11] + C3[3] * z * (2 * zz - 3 * xx - 3 * yy) * sh[..., 12] +
                     C3[4] * x * (4 * zz - xx - yy) * sh[..., 13] + C3[5] * z * (xx - yy) * sh[..., 14] +
                     C3[6] * x * (xx - 3 * yy) * sh[..., 15])
    return r


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_sh_colors_match_eval_sh(deg):
    cloud, cams = synth.make_config("c3", P=400)
    cloud.sh_degree = deg
    cam = cams[1]
    f = O.forward_from(cloud, cam, f32=False)
    vis = f.radii > 0
    d = cloud.means3D.astype(np.float64) - cam.campos.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sh = cloud.shs.astype(np.float64).transpose(0, 2, 1)      # [P,3,M] like the reference's shs_view
    want = np.maximum(_eval_sh_numpy(deg, sh, d) + 0.5, 0.0)
    assert vis.sum() > 50
    assert np.allclose(f.rgb[vis], want[vis], atol=3e-7)  # the oracle keeps the fp32 SH constants
    assert np.array_equal(f.clamped[vis].astype(bool), (_eval_sh_numpy(deg, sh, d) + 0.5 < 0)[vis])


def test_cov3d_matches_build_scaling_rotation():
    cloud, cams = synth.make_config("c3", P=300)
    f = O.forward_from(cloud, cams[0], f32=False, scale_modifier=1.3)
    q = cloud.rotations.astype(np.float64)
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R = np.zeros((len(q), 3, 3))     # utils/general_utils.py:78-99 build_rotation (row-major, normalised input)
    R[:, 0, 0] = 1 - 2 * (y * y + z * z); R[:, 0, 1] = 2 * (x * y - r * z); R[:, 0, 2] = 2 * (x * z + r * y)
    R[:, 1, 0] = 2 * (x * y + r * z); R[:, 1, 1] = 1 - 2 * (x * x + z * z); R[:, 1, 2] = 2 * (y * z - r * x)
    R[:, 2, 0] = 2 * (x * z - r * y); R[:, 2, 1] = 2 * (y * z + r * x); R[:, 2, 2] = 1 - 2 * (x * x + y * y)
    S = float(np.float32(1.3)) * cloud.scales.astype(np.float64)
    L = R * S[:, None, :]                                       # R @ diag(s)
    Sigma = L @ L.transpose(0, 2, 1)
    want = np.stack([Sigma[:, 0, 0], Sigma[:, 0, 1], Sigma[:, 0, 2], Sigma[:, 1, 1], Sigma[:, 1, 2], Sigma[:, 2, 2]], 1)
    vis = f.depths > 0.2
    assert np.allclose(f.cov3D[vis], want[vis], rtol=1e-9, atol=1e-12)


def test_fp32_oracle_agrees_with_fp64_oracle():
    cloud, cams = synth.make_config("c3", P=20_000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 160, 120, 61.0)[3]
    a = O.forward_from(cloud, cam, bg=(0.1, 0.2, 0.3), f32=True)
    b = O.forward_from(cloud, cam, bg=(0.1, 0.2, 0.3), f32=False)
    assert (a.radii != b.radii).mean() < 1e-3
    assert np.mean(np.abs(a.color - b.color) > 1e-4) < 1e-3
    dL = np.random.default_rng(0).uniform(size=(3, 120, 160)).astype(np.float32)
    ga, gb = a.backward(dL), b.backward(dL)
    for k in ["dmean3D", "dmean2D", "dopacity", "dscale", "drot", "dsh"]:
        err = np.linalg.norm(ga[k] - gb[k]) / np.linalg.norm(gb[k])
        assert err < 5e-3, (k, err)


def test_stable_order_for_equal_depths():
    cam = _cam(32, 32)
    # three coincident centres -> identical depth bits; list order must be ascending Gaussian index
    cloud = _cloud([[0, 0, 0]] * 3, [[0.2] * 3] * 3, [[1, 0, 0, 0]] * 3, [[0.3]] * 3, rgb_dc=[[1, 0, 0], [0, 1, 0], [0, 0, 1]])
    f = O.forward_from(cloud, cam)
    for t in range(f.ranges.shape[0]):
        lst = list(f.point_list[f.ranges[t, 0]:f.ranges[t, 1]])
        assert lst == sorted(lst)


def _loss_and_grads(cloud, cam, G, bg):
    f = O.forward_from(cloud, cam, bg=bg, f32=False)
    loss = float((f.color * G).sum())
    g = f.backward(G.astype(np.float32))
    nc = f.n_contrib.copy(); radii = f.radii.copy()
    f.close()
    return loss, g, nc, radii


def test_gradients_match_fp64_finite_differences():
    """Directional finite differences of loss = sum(color * G) in fp64 for every differentiable input."""
    rng = np.random.default_rng(42)
    cam = _cam(40, 32, fovy=45.0)
    P = 24
    xyz = rng.uniform(-0.6, 0.6, (P, 3))
    sc = np.exp(rng.normal(math.log(0.12), 0.3, (P, 3)))
    q = rng.standard_normal((P, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    op = rng.uniform(0.2, 0.9, (P, 1))
    sh = rng.standard_normal((P, 16, 3)) * 0.3
    sh[:, 0, :] += 1.0
    cloud = synth.Cloud(xyz.astype(np.float32), sc.astype(np.float32), q.astype(np.float32), op.astype(np.float32),
                        sh.astype(np.float32), 3)
    G = rng.uniform(size=(3, 32, 40)).astype(np.float32).astype(np.float64)
    bg = (0.3, 0.1, 0.6)
    loss0, g, nc0, radii0 = _loss_and_grads(cloud, cam, G, bg)
    fields = [("means3D", "dmean3D"), ("scales", "dscale"), ("rotations", "drot"), ("opacities", "dopacity"),
              ("shs", "dsh")]
    for field, gname in fields:
        ok = tried = 0
        for trial in range(12):
            base = getattr(cloud, field)
            d = rng.standard_normal(base.shape)
            d /= np.linalg.norm(d)
            for eps in (3e-5, 1e-5):
                # inputs are float32 arrays: perturb with a float32-representable step and use the step actually taken
                plus = (base.astype(np.float64) + eps * d).astype(np.float32)
                minus = (base.astype(np.float64) - eps * d).astype(np.float32)
                step = (plus.astype(np.float64) - minus.astype(np.float64))
                l1, _, n1, r1 = _loss_and_grads(synth.Cloud(**{**cloud.__dict__, field: plus}), cam, G, bg)
                l2, _, n2, r2 = _loss_and_grads(synth.Cloud(**{**cloud.__dict__, field: minus}), cam, G, bg)
                # the rasterizer is piecewise smooth: radius steps, the alpha<1/255 skip and the T<1e-4 stop are
                # jumps; a direction is only usable when the perturbation crosses none that we can detect
                if not (np.array_equal(r1, radii0) and np.array_equal(r2, radii0) and np.array_equal(n1, nc0)
                        and np.array_equal(n2, nc0)):
                    continue
                tried += 1
                ana = float((g[gname].reshape(base.shape) * step).sum())
                if abs((l1 - l2) - ana) <= 2e-4 * abs(ana) + 1e-12:
                    ok += 1
        # undetected alpha<1/255 crossings of non-final contributors can still spoil a direction; most must agree
        assert tried >= 6 and ok >= 0.7 * tried, (field, ok, tried)
    # dmean2D is the gradient w.r.t. the NDC-scaled screen position: checked through its chain into dmean3D above;
    # its z component is identically zero and invisible Gaussians get exact zeros
    assert np.all(g["dmean2D"][:, 2] == 0)


def test_apply_weights_counts():
    cloud, cams = synth.make_config("c3", P=3000)
    cam = synth.ring_cameras(8, 4.5, 15.0, 96, 64, 61.0)[0]
    f = O.forward_from(cloud, cam, colors_precomp=np.zeros((3000, 3), np.float32))
    mask = np.ones((1, 64, 96), np.float32)
    w = np.zeros((3000, 1), np.float32); cnt = np.zeros((3000, 1), np.int32)
    f.apply_weights(w, cnt, mask)
    # with an all-ones single-channel mask, weight == count == number of pixels the splat is blended into
    assert np.array_equal(w[:, 0], cnt[:, 0].astype(np.float32))
    assert cnt.sum() == f.hits
    assert cnt[f.radii == 0].sum() == 0


def test_precomputed_colour_and_covariance_paths_of_the_oracle():
    """The two alternative input paths (Appendix A item 16: colors_precomp is live in GaussianEditor's mask render;
    cov3D_precomp is never used there but part of the API): precomputed inputs that equal what the oracle derives
    itself must give the same image, and the colour gradient must be the plain blending weight sum (closed form:
    dL/dcolor_i = sum_pixels alpha_i * T_i * G), independent of the SH machinery."""
    cloud, cams = synth.make_config("c3", P=1500)
    cam = synth.ring_cameras(8, 4.5, 15.0, 112, 80, 61.0)[3]
    bg = (0.2, 0.4, 0.1)
    base = O.forward_from(cloud, cam, bg, f32=False)
    vis = base.radii > 0
    # colours: feed the oracle's own SH->RGB result back as precomputed colours
    rgb = np.where(vis[:, None], base.rgb, 0.0).astype(np.float32)
    pc = O.forward_from(cloud, cam, bg, f32=False, colors_precomp=rgb)
    assert np.array_equal(pc.radii, base.radii) and np.array_equal(pc.point_list, base.point_list)
    assert np.allclose(pc.color, base.color, atol=2e-7)        # rgb went through float32 once
    # covariance: feed cov3D back
    cov = np.where(vis[:, None], base.cov3D, 0.0).astype(np.float32)
    cv = O.forward_from(cloud, cam, bg, f32=False, cov3D_precomp=cov, scales=None, rotations=None)
    assert (cv.radii != base.radii).mean() <= 2e-3            # cov3D rounded to float32 moves a radius step rarely
    same = cv.radii == base.radii
    assert np.allclose(cv.conic_opacity[same & vis], base.conic_opacity[same & vis], rtol=2e-4, atol=1e-9)
    # colour gradient is linear in G with the blending weights as coefficients: doubling G doubles it exactly, and a
    # one-hot G on a pixel gives alpha*T of the splats that cover it, which sum with final_T to 1 (energy conservation)
    H, W = cam.image_height, cam.image_width
    G = np.zeros((3, H, W), np.float32)
    py, px = H // 2, W // 2
    G[0, py, px] = 1.0
    g = pc.backward(G)
    weights = g["dcolor"][:, 0]
    assert np.all(weights >= 0) and abs(weights.sum() + pc.final_T[py, px] - 1.0) <= 1e-9
    assert np.all(g["dcolor"][:, 1:] == 0)
    g2 = pc.backward(2.0 * G)
    assert np.allclose(g2["dcolor"], 2.0 * g["dcolor"], rtol=0, atol=0)
    base.close(); pc.close(); cv.close()


@pytest.mark.parametrize("W,H,scene", [(333, 201, "c3"), (4160, 48, "c3"), (7, 5, "c3"), (333, 201, "adversarial")])
def test_binning_restatement_equals_the_oracle(W, H, scene):
    """tests/util.bin_reference (the numpy binning the GPU shape sweep compares against) rebuilds the fp32 oracle's own
    tiles_touched, R, ranges and point_list bit for bit from the oracle's means2D, radii and depths -- incl. a partial
    last tile row and column, a frame with > 256 tile columns, a single tile, and groups of bit-equal depths."""
    from util import adversarial_scene, axis_camera, bin_reference
    if scene == "c3":
        cloud, _ = synth.make_config("c3", P=20_000)
        cam = synth.ring_cameras(8, 4.5, 15.0, W, H, 61.0)[5]
    else:
        cloud, cls = adversarial_scene()
        cam = axis_camera(W, H)
    f = O.forward_from(cloud, cam, render=False)
    got = bin_reference(f.means2D, f.radii, f.depths, W, H)
    assert got["R"] == f.num_rendered > 0
    assert np.array_equal(got["tiles_touched"], f.tiles_touched)
    assert np.array_equal(got["ranges"], f.ranges)
    assert np.array_equal(got["point_list"], f.point_list)
    if scene == "adversarial":   # the tie-break by Gaussian index is exercised
        d = f.depths[f.point_list]
        assert np.sum(d[1:] == d[:-1]) >= 50
    f.close()
